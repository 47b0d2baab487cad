// nn.cu -- the policy / value / uncertainty ResNet of the reference as a device agent.
//
// Replaces `impl Agent<Env> for Net` (takzero/src/network/net6_simhash.rs:259-324 and its
// N = 4 / N = 5 siblings): board -> input planes (network/repr.rs:169-228) -> conv tower
// (net6_simhash.rs:43-72, residual.rs) -> policy conv + legal-logit gather (:74-86,277-306),
// value / UBE heads (:88-119) and the uncertainty combine (:309-317), without libtorch; and
// `Net::load` (network/mod.rs:16-35) with the per-move reload of selfplay/src/main.rs:107 as a
// weight GENERATION: fold + arrange on the GPU into the inactive one of two weight sets, optionally
// broadcast over NCCL (comm.cu), swapped in between two moves.
// The 3x3 convolutions run on tcgen05 (conv_tcgen05.cuh); everything else here is small.
#include <math.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <string>
#include <type_traits>
#include <utility>
#include <vector>

#include "comm.cuh"
#include "conv_tcgen05.cuh"
#include "encode.cuh"
#include "nn.cuh"
#include "planes.cuh"
#include "rnd.cuh"
#include "rules.cuh"

#define WPB TZ_WARPS_PER_BLOCK
#define FILTERS 256
#define CIN_PAD 64
#define SET_HEADER_BYTES 256
#define SET_MAGIC 0x53575a54u  // "TZWS"
#define NOVELTY_BYTES ((size_t)1 << 29)        // the 2^32-bit novelty set (bitvec.bin)
#define NOVELTY_STAGE_BYTES ((size_t)8 << 20)  // each of the two pinned chunks a pageable set image goes through
#define NOVELTY_MAGIC 0x53535a54u              // "TZSS": header of a broadcast novelty set

// Byte offsets inside one weight set (a single device allocation, so that a generation travels as ONE broadcast):
// [header 256 B][per convolution: blocks in the shared-memory image the tensor core reads, then 256 f32 biases]
// [value / UBE 1x1 weights 2 x 256 f32][head_misc 76 f32].  A function of (board size, residual blocks) only.
struct SetLayout {
    int layers = 0;  // 2 * blocks + 2: input convolution, tower, policy convolution
    int cin_pad[conv::MAX_LAYERS];
    size_t w[conv::MAX_LAYERS], b[conv::MAX_LAYERS];
    size_t head_w = 0, head_misc = 0, total = 0;
};
// Float offsets inside the raw f32 staging buffer the fold kernels read (root of a generation only): per convolution
// the PyTorch-layout weight [cout][cin][3][3], then either the four BatchNorm vectors (weight, bias, running_mean,
// running_var; 256 each) or (policy) the convolution bias; then value / UBE 1x1 weights and head_misc.
struct RawLayout {
    int cout[conv::MAX_LAYERS], cin[conv::MAX_LAYERS], has_bn[conv::MAX_LAYERS];
    size_t w[conv::MAX_LAYERS], aux[conv::MAX_LAYERS];
    size_t heads = 0, total = 0;
};

struct NnState {
    int n = 0, blocks = 0;
    int in_channels = 0, out_channels = 0;
    int max_positions = 0;
    size_t rows_set = 0;  // rows per chunk plane of one activation set (one chunk of positions)
    int pack = 0;         // positions per CTA tile of the packed small-batch layout (conv::Params::pack), 0: never
    int chunk_min_tiles = 0;   // least pair tiles the network runs through all layers at a time (conv_tcgen05.cuh)
    int chunk_tiles = 0, max_chunks = 0;  // bounds: pair tiles of one chunk, chunks of one launch
    // weights: two sets, `active` is the one new launches read (-1: none yet)
    SetLayout lay;
    RawLayout raw;
    uint8_t* wset[2] = {nullptr, nullptr};
    int set_f16[2] = {0, 0};  // 16-bit type of each set's weights (and of the activations of launches that use it)
    int active = -1;
    unsigned long long generation = 0;
    float* raw_dev = nullptr;  // raw f32 tensors of the generation being folded
    float* raw_pin = nullptr;  // pinned host staging of the same (tensors that come from pageable memory)
    float* head_pin = nullptr; // pinned staging of the small head tensors (always assembled on the host)
    struct DirectCopy {
        size_t off, count;
        const float* src;
    };
    std::vector<DirectCopy> direct;  // this generation's tensors that already sit in pinned memory: copied from there
    cudaStream_t wstream = nullptr;  // uploads, folds and broadcasts run beside the search stream
    cudaEvent_t ev_ready = nullptr;  // wstream: the new set is complete
    cudaEvent_t ev_swap = nullptr;   // search stream: everything enqueued before the last swap (the readers of the
                                     // set that is inactive now)
    cudaEvent_t ev_h2d = nullptr;    // wstream: raw_pin has been read
    cudaEvent_t ev_gen[2] = {nullptr, nullptr};  // wstream: start / end of the last generation (its device time)
    bool swap_recorded = false, h2d_recorded = false, gen_timed = false;
    // chunk-planar activations (conv_tcgen05.cuh): [channels / 8][rows][8]
    __nv_bfloat16* act_x = nullptr;   // [2 sets][32][rows_set][8]  residual stream (even / odd chunks)
    __nv_bfloat16* act_t = nullptr;   // [2 sets][32][rows_set][8]  middle of a residual block
    __nv_bfloat16* tune_buf[3] = {nullptr, nullptr, nullptr};  // tuning hook only
    float* head_feat = nullptr;       // [max_positions * n*n][2] value / UBE 1x1 convolution outputs per row
    uint16_t* perm = nullptr;         // [max_positions][M] host action lists grouped by square (tz_evaluate only)
    uint4* masks = nullptr;           // [n*n][9] disable-output-lane masks (conv_tcgen05.cuh)
    int novelty = 0;                  // which hash indexes the set: 0 none yet, 1 SimHash, 2 LCG hash (last one set)
    float* lcghash_init = nullptr;    // [C][N][N] (net4_lcghash.rs:131-137), optional
    float* simhash_matrix = nullptr;  // [C*N*N][32] (net6_simhash.rs:136-139), optional
    uint32_t* simhash_set = nullptr;  // 2^32-bit set (bitvec.bin), optional; absent = empty set
    uint32_t* simhash_set_alloc = nullptr;
    uint32_t* simhash_idx = nullptr;  // [max_positions] hash index of each queued position
    // set generations (tz_broadcast_novelty_set), all created by the first one: the inactive set the next generation
    // is written into (swapped with simhash_set_alloc), the broadcast header ([0..3] magic, hash kind, board size;
    // [4] this rank's mismatch flag), the pinned chunks of pageable images and their events
    uint32_t* set_spare = nullptr;
    uint32_t* set_hdr = nullptr;
    unsigned char* set_pin = nullptr;
    cudaEvent_t ev_stage[2] = {nullptr, nullptr};  // wstream: chunk k of set_pin has been read
    bool stage_used[2] = {false, false};
    cudaEvent_t ev_marks = nullptr;  // search stream: the marks a generation copies (or keeps) have landed
    size_t progress_len = 0;
    unsigned* progress = nullptr;     // [chunks][pair tiles] tile-completion counters of the fused launch, then
                                      // [chunks] chunk-completion counters
    int max_pairs = 74;               // CTA pairs that can be resident at once (cooperative launch bound)
    int fused = 1;                    // 1: the network is one multi-layer launch; 0 (debug mode): one launch per layer
    int cfg_chunk_tiles = -1;         // the tz_debug_network_mode chunking this state was sized with (-1 = default)
    int layer_limit = -1;             // debug: stop the tower after this many convolutions
    std::vector<void*> allocs;
    int sm_count = 148;
};

bool nn_ready(const tz_handle* h) { return h->nn != nullptr && h->nn->active >= 0; }

void nn_free(tz_handle* h) {
    NnState* s = h->nn;
    if (!s) return;
    if (s->wstream) cudaStreamSynchronize(s->wstream);
    for (void* p : s->allocs) cudaFree(p);
    if (s->raw_pin) cudaFreeHost(s->raw_pin);
    if (s->head_pin) cudaFreeHost(s->head_pin);
    if (s->set_pin) cudaFreeHost(s->set_pin);
    for (cudaEvent_t e : {s->ev_ready, s->ev_swap, s->ev_h2d, s->ev_gen[0], s->ev_gen[1], s->ev_stage[0], s->ev_stage[1],
                          s->ev_marks})
        if (e) cudaEventDestroy(e);
    if (s->wstream) cudaStreamDestroy(s->wstream);
    delete s;
    h->nn = nullptr;
    h->d.nn_head_feat = nullptr;
    h->d.nn_head_misc = nullptr;
    h->d.nn_novelty_set = nullptr;
    h->d.nn_novelty_idx = nullptr;
    h->d.nn_rnd_unc = nullptr;
    rnd_free(h);
}

// ---- input planes (network/repr.rs:169-228), parity hook -------------------------------------------

// One warp per position.  out_f32: [count][C][N][N] exactly like `game_repr`.  (The network itself never stores its
// input planes: the first convolution's A producer encodes them straight into shared memory, conv_tcgen05.cuh.)
__global__ void __launch_bounds__(32 * WPB) k_encode(const TzState* states, int count, int n, int half_komi,
                                                      float* out_f32) {
    __shared__ TzState s_state[WPB];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q = blockIdx.x * WPB + warp;
    if (q >= count) return;
    TzState* st = &s_state[warp];
    warp_load_state(st, &states[q], lane);
    const int C = 2 * (2 * n + 5) + 2;
    warp_encode_planes(st, n, half_komi, out_f32 + (size_t)q * C * n * n, lane);
}

// parity hook for the 16-bit planes the first convolution's A producer builds (same device function): one thread
// per (position, square), the 64 channels widened to f32: out[count][N*N][64]
__global__ void k_encode16(const TzState* states, int count, int n, int f16, float* out) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int nn = n * n;
    if (idx >= count * nn) return;
    const int q = idx / nn, sq = idx - q * nn;
    const uint8_t* st = reinterpret_cast<const uint8_t*>(states + q);
    const uint64_t stack = *reinterpret_cast<const uint64_t*>(st + 8 * sq);
    const uint4 tail = *reinterpret_cast<const uint4*>(st + 368);
    enc::PositionScalars ps;
    ps.s01 = tail.y;
    ps.s23 = tail.z;
    ps.s45 = tail.w;
    uint4 px[8];
    enc::encode_square16(stack, st[288 + sq], st[324 + sq], st[360], ps, n, f16, px);
    const uint32_t* w = reinterpret_cast<const uint32_t*>(px);
    for (int p = 0; p < 32; p++) {
        const float2 v = conv::unpack16(w[p], f16);
        out[(size_t)idx * 64 + 2 * p] = v.x;
        out[(size_t)idx * 64 + 2 * p + 1] = v.y;
    }
}

// ---- SimHash novelty index (net6_simhash.rs:203-234 `get_indices`) ---------------------------------

// One warp, lane = hash bit: dot of the f32 planes (side-to-move plane zeroed, built in x) with column `lane` of the
// [C*N*N][32] matrix; bit set when the dot is >= 0; index = sum of 2^bit, in every lane.
__device__ __forceinline__ uint32_t warp_simhash(const TzState* st, int n, int half_komi, const float* matrix, float* x,
                                                 int lane) {
    const int nn = n * n, C = 2 * (2 * n + 3 + 2) + 2;
    warp_fill_planes(x, st, n, half_komi, lane, true);
    float dot = 0.0f;
    const int total = C * nn;
    for (int j = 0; j < total; j++) dot = fmaf(x[j], matrix[(size_t)j * 32 + lane], dot);
    return __ballot_sync(0xffffffffu, !(dot < 0.0f));
}

// ---- LCG-hash novelty index (net4_lcghash.rs:203-241 `get_indices`) -------------------------------------
// planes * lcghash_init (f32, elementwise) reinterpreted as i32, folded with the 64-bit LCG
// acc = acc * 6364136223846793005 + 1 + v  along the columns, then the rows, then the channels (wrapping i64);
// index = |acc| >> 31.  Integer work: bit-exact.  One warp (x: the planes, rows: C * N folds); the index is valid in
// lane 0.
__device__ __forceinline__ uint32_t warp_lcghash(const TzState* st, int n, int half_komi, const float* init, float* x,
                                                 unsigned long long* rows, int lane) {
    const int C = 2 * (2 * n + 3 + 2) + 2;
    warp_fill_planes(x, st, n, half_komi, lane, false);
    const unsigned long long MUL = 6364136223846793005ull;
    for (int cr = lane; cr < C * n; cr += 32) {  // (channel, row): fold the columns
        unsigned long long acc = 0;
        for (int j = 0; j < n; j++) {
            const int at = cr * n + j;
            const int v = __float_as_int(__fmul_rn(x[at], init[at]));
            acc = acc * MUL + 1ull + (unsigned long long)(long long)v;
        }
        rows[cr] = acc;
    }
    __syncwarp();
    for (int c = lane; c < C; c += 32) {  // channel: fold the rows (in place: slot c * n)
        unsigned long long acc = 0;
        for (int r = 0; r < n; r++) acc = acc * MUL + 1ull + rows[c * n + r];
        __syncwarp();
        rows[c * n] = acc;
    }
    __syncwarp();
    uint32_t index = 0;
    if (lane == 0) {
        unsigned long long acc = 0;
        for (int c = 0; c < C; c++) acc = acc * MUL + 1ull + rows[c * n];
        long long sacc = (long long)acc;
        if (sacc < 0) sacc = -sacc;  // i64::MIN stays negative, as a wrapping abs does
        index = (uint32_t)((unsigned long long)sacc >> 31);
    }
    return index;
}

// One warp per position: the hash index of every position.
__global__ void __launch_bounds__(32 * WPB) k_simhash(const TzState* states, const int* count_ptr, int count_max, int n,
                                                       int half_komi, const float* matrix, uint32_t* out_idx) {
    __shared__ TzState s_state[WPB];
    __shared__ float s_planes[WPB][36 * 36];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q = blockIdx.x * WPB + warp;
    const int count = count_ptr ? *count_ptr : count_max;
    if (q >= count) return;
    TzState* st = &s_state[warp];
    warp_load_state(st, &states[q], lane);
    const uint32_t bits = warp_simhash(st, n, half_komi, matrix, s_planes[warp], lane);
    if (lane == 0) out_idx[q] = bits;
}

__global__ void __launch_bounds__(32 * WPB) k_lcghash(const TzState* states, const int* count_ptr, int count_max, int n,
                                                       int half_komi, const float* init, uint32_t* out_idx) {
    __shared__ TzState s_state[WPB];
    __shared__ float s_planes[WPB][36 * 36];
    __shared__ unsigned long long s_rows[WPB][36 * 6];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q = blockIdx.x * WPB + warp;
    const int count = count_ptr ? *count_ptr : count_max;
    if (q >= count) return;
    TzState* st = &s_state[warp];
    warp_load_state(st, &states[q], lane);
    const uint32_t index = warp_lcghash(st, n, half_komi, init, s_planes[warp], s_rows[warp], lane);
    if (lane == 0) out_idx[q] = index;
}

// tz_update_counts_buffer: one warp per example of a training batch.  The example's target (resolved as
// k_training_batch does) is read from the ring, transformed by its symmetry, hashed with the handle's hash
// (kind 1 SimHash: w = matrix, 2 LCG: w = multipliers) and its bit ORed into the set.
__global__ void __launch_bounds__(32 * WPB) k_mark_batch(TzTargetRing R, int n, int half_komi, int batch,
                                                          const unsigned long long* indices, const int* symmetry,
                                                          int augment, unsigned long long seed, unsigned long long size,
                                                          unsigned long long first, int kind, const float* w,
                                                          uint32_t* set) {
    __shared__ TzState s_src[WPB], s_dst[WPB];
    __shared__ float s_planes[WPB][36 * 36];
    __shared__ unsigned long long s_rows[WPB][36 * 6];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int b = blockIdx.x * WPB + warp;
    if (b >= batch) return;
    unsigned long long idx;
    int t;
    batch_example(indices, symmetry, augment, seed, size, b, &idx, &t);
    const unsigned long long slot = (first + idx) % R.cap;
    warp_load_state(&s_src[warp], &R.env[slot], lane);
    warp_symmetric_state(&s_dst[warp], &s_src[warp], t, n, lane);
    const uint32_t index = kind == 2 ? warp_lcghash(&s_dst[warp], n, half_komi, w, s_planes[warp], s_rows[warp], lane)
                                     : warp_simhash(&s_dst[warp], n, half_komi, w, s_planes[warp], lane);
    if (lane == 0) atomicOr(&set[index >> 5], 1u << (index & 31));
}

// ---- host-supplied positions (tz_evaluate): what k_select provides for queued leaves ------------------------

// One warp per position: the per-position input-plane words into the device copy of the state (encode.cuh
// `store_position_scalars`) and the action list grouped by square: ranges[q][square] = first | count << 16 into perm[q][...], which lists the
// indices of the moves that start on each square (the epilogue of the policy convolution gathers by square).
// Host lists may come in any order and may hold impossible moves; those are skipped (their logit stays 0).
__global__ void __launch_bounds__(32 * WPB) k_prepare_eval(TzState* states, int count, int n, int half_komi, int f16,
                                                            const uint16_t* actions, const int* n_actions, int M,
                                                            uint32_t* ranges, uint16_t* perm) {
    __shared__ TzState s_state[WPB];
    __shared__ int s_cnt[WPB][TZ_MAX_SQ], s_cur[WPB][TZ_MAX_SQ];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q = blockIdx.x * WPB + warp;
    if (q >= count) return;
    const int nn = n * n;
    TzState* st = &s_state[warp];
    warp_load_state(st, &states[q], lane);
    const TzBoards b = warp_boards(st, nn, lane);
    if (lane == 0) enc::store_position_scalars(st, __popcll(b.flat[0]) - __popcll(b.flat[1]), n, half_komi, f16);
    __syncwarp();
    if (lane == 0) *reinterpret_cast<uint4*>(reinterpret_cast<uint8_t*>(&states[q]) + 368) =
                       *reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(st) + 368);
    for (int sq = lane; sq < TZ_MAX_SQ; sq += 32) s_cnt[warp][sq] = 0;
    __syncwarp();
    const int cnt = n_actions[q];
    const uint16_t* a = actions + (size_t)q * M;
    for (int i = lane; i < cnt; i += 32) {
        const int col = a[i] & 7, row = (a[i] >> 3) & 7;
        if (row < n && col < n) atomicAdd(&s_cnt[warp][row * n + col], 1);
    }
    __syncwarp();
    if (lane == 0) {
        int off = 0;
        for (int sq = 0; sq < nn; sq++) {
            s_cur[warp][sq] = off;
            ranges[(size_t)q * TZ_MAX_SQ + sq] = (uint32_t)off | ((uint32_t)s_cnt[warp][sq] << 16);
            off += s_cnt[warp][sq];
        }
    }
    __syncwarp();
    for (int i = lane; i < cnt; i += 32) {
        const int col = a[i] & 7, row = (a[i] >> 3) & 7;
        if (row < n && col < n) perm[(size_t)q * M + atomicAdd(&s_cur[warp][row * n + col], 1)] = (uint16_t)i;
    }
}

// One warp per position: the heads' last step (encode.cuh `warp_heads`), for callers that want value / variance
// arrays (tz_evaluate); the search does the same inside k_expand.
__global__ void __launch_bounds__(32 * WPB) k_heads(const float* head_feat, const float* head_misc, int count, int n,
                                                     const uint32_t* novelty_set, const uint32_t* novelty_idx,
                                                     const float* rnd_unc, float* out_value, float* out_variance) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q = blockIdx.x * WPB + warp;
    if (q >= count) return;
    float value, variance;
    enc::warp_heads(head_feat, head_misc, novelty_set, novelty_idx, rnd_unc, q, n * n, lane, &value, &variance);
    if (lane == 0) {
        out_value[q] = value;
        out_variance[q] = variance;
    }
}

// ---- weights: fold + arrange on the device ---------------------------------------------------------------

struct FoldLayer {
    long long w, aux;      // float offsets into the raw buffer: weight [cout][cin][3][3]; BN vectors or conv bias
    long long out_w, out_b;  // byte offsets into the weight set
    int cout, cin, cin_pad, has_bn;
};
struct FoldParams {
    FoldLayer L[conv::MAX_LAYERS];
    int layers;
    const float* raw;
    uint8_t* set;
    int f16;
};

// BatchNorm (eval mode, eps 1e-5 = tch BatchNormConfig::default) folded into the convolution, in the operation order
// of a plain f32 host loop: scale = bn_w * (1 / sqrt(var + eps)); w' = w * scale; bias = bn_b - mean * scale
// (+ conv_bias * scale)
__device__ __forceinline__ float fold_scale(const FoldLayer& L, const float* raw, int co) {
    if (!L.has_bn) return 1.0f;
    const float* bn = raw + L.aux;
    const float inv = __fdiv_rn(1.0f, __fsqrt_rn(__fadd_rn(bn[3 * FILTERS + co], 1e-5f)));
    return __fmul_rn(bn[co], inv);
}

// grid (elements / 256, layers): one thread per 16-bit element of the arranged weights.  Output image per layer:
// [cin_pad/64 k-blocks][9 taps, centre first][2 N halves][8 k-chunks][128 n][8] -- one contiguous 16 KB block per
// (k-block, tap, CTA of the pair), exactly what a B stage of the convolution kernel holds.
__global__ void k_fold_weights(const __grid_constant__ FoldParams p) {
    const FoldLayer& L = p.L[blockIdx.y];
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    const long long total = (long long)(L.cin_pad / 64) * 9 * 16384;
    if (idx >= total) return;
    const int e = (int)(idx & 7), nrow = (int)((idx >> 3) & 127), kc = (int)((idx >> 10) & 7), half = (int)((idx >> 13) & 1);
    const int rest = (int)(idx >> 14), ti = rest % 9, kb = rest / 9;
    const int tap = ti == 0 ? 4 : (ti <= 4 ? ti - 1 : ti);  // tap = ky * 3 + kx; the kernel consumes the centre first
    const int co = half * 128 + nrow, ci = kb * 64 + kc * 8 + e;
    float v = 0.0f;
    if (co < L.cout && ci < L.cin) v = __fmul_rn(p.raw[L.w + ((long long)co * L.cin + ci) * 9 + tap], fold_scale(L, p.raw, co));
    uint16_t* out = reinterpret_cast<uint16_t*>(p.set + L.out_w);
    if (p.f16) {
        const __half hv = __float2half_rn(v);
        out[idx] = *reinterpret_cast<const uint16_t*>(&hv);
    } else {
        const __nv_bfloat16 bv = __float2bfloat16_rn(v);
        out[idx] = *reinterpret_cast<const uint16_t*>(&bv);
    }
}

// grid (layers), 256 threads: the folded bias of every output channel
__global__ void k_fold_bias(const __grid_constant__ FoldParams p) {
    const FoldLayer& L = p.L[blockIdx.x];
    const int co = threadIdx.x;
    float bias = 0.0f;
    if (co < L.cout) {
        const float scale = fold_scale(L, p.raw, co);
        if (L.has_bn) {
            const float* bn = p.raw + L.aux;
            bias = __fsub_rn(bn[FILTERS + co], __fmul_rn(bn[2 * FILTERS + co], scale));
        } else if (L.aux >= 0) {
            bias = __fadd_rn(bias, __fmul_rn(p.raw[L.aux + co], scale));
        }
    }
    reinterpret_cast<float*>(p.set + L.out_b)[co] = bias;
}

__global__ void k_set_header(uint8_t* set, uint32_t n, uint32_t blocks, uint32_t f16, unsigned long long generation) {
    uint32_t* h = reinterpret_cast<uint32_t*>(set);
    h[0] = SET_MAGIC;
    h[1] = n;
    h[2] = blocks;
    h[3] = f16;
    h[4] = (uint32_t)generation;
    h[5] = (uint32_t)(generation >> 32);
}

// after a broadcast: the set that arrived must describe this handle's network
__global__ void k_check_header(const uint8_t* set, uint32_t n, uint32_t blocks, uint32_t f16, uint32_t* status) {
    const uint32_t* h = reinterpret_cast<const uint32_t*>(set);
    if (h[0] != SET_MAGIC || h[1] != n || h[2] != blocks || h[3] != f16) atomicOr(status, TZ_ERR_WEIGHTS_MISMATCH);
}

// ---- weights: host side ----------------------------------------------------------------------------------------

struct HostTensor {
    std::string name;
    const float* data;
    std::vector<long long> shape;
    size_t numel() const {
        size_t k = 1;
        for (long long s : shape) k *= (size_t)s;
        return k;
    }
};

static const HostTensor* find(const std::vector<HostTensor>& ts, const std::string& name) {
    for (const HostTensor& t : ts)
        if (t.name == name) return &t;
    return nullptr;
}

// Upper bounds of what conv::Schedule::init derives from a device-side count <= count_max: number of chunks and
// pair tiles of one chunk (a chunk has fewer than 2 * chunk_min_tiles tiles, + rounding).  The activation sets and
// the progress counters are sized with these.
struct ChunkBounds {
    int chunks, chunk_tiles;
};
static ChunkBounds chunk_bounds(int count_max, int nn, int chunk_min_tiles) {
    const int all_tiles = (int)(((long long)count_max * nn + 2 * conv::TILE_M - 1) / (2 * conv::TILE_M));
    ChunkBounds b;
    b.chunks = all_tiles >= 2LL * chunk_min_tiles ? all_tiles / chunk_min_tiles : 1;
    b.chunk_tiles = b.chunks > 1 ? 2 * chunk_min_tiles + 2 : (all_tiles > 0 ? all_tiles : 1);
    return b;
}

static thread_local char g_nn_err[256] = "";
const char* nn_last_error() { return g_nn_err; }
#define NN_FAIL(code, ...)                              \
    do {                                                \
        snprintf(g_nn_err, sizeof(g_nn_err), __VA_ARGS__); \
        return code;                                    \
    } while (0)

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

static void make_layouts(int n, int blocks, SetLayout* lay, RawLayout* raw) {
    const int cin0 = 2 * (2 * n + 3 + 2) + 2, cout_p = 3 + 4 * ((1 << n) - 2);
    lay->layers = 2 * blocks + 2;
    size_t off = SET_HEADER_BYTES, roff = 0;
    for (int l = 0; l < lay->layers; l++) {
        const bool first = l == 0, last = l == lay->layers - 1;
        lay->cin_pad[l] = first ? CIN_PAD : FILTERS;
        lay->w[l] = off;
        off += (size_t)(lay->cin_pad[l] / 64) * 9 * 16384 * 2;
        lay->b[l] = off;
        off += FILTERS * sizeof(float);
        raw->cout[l] = last ? cout_p : FILTERS;
        raw->cin[l] = first ? cin0 : FILTERS;
        raw->has_bn[l] = last ? 0 : 1;
        raw->w[l] = roff;
        roff += (size_t)raw->cout[l] * raw->cin[l] * 9;
        raw->aux[l] = roff;
        roff += last ? (size_t)FILTERS : (size_t)4 * FILTERS;  // policy: conv bias (padded to 256)
    }
    lay->head_w = off;
    off += 2 * FILTERS * sizeof(float);
    lay->head_misc = off;
    off += 76 * sizeof(float);
    lay->total = align_up(off, 256);
    raw->heads = roff;
    roff += 2 * FILTERS + 76;
    raw->total = roff;
}

// names and shapes of a complete model for an N x N board; *blocks from the names (16 for net4 / net6, 20 for net5)
static int validate_tensors(const std::vector<HostTensor>& ts, int n, int* blocks) {
    const long long n0 = n, cin0 = 2 * (2 * n0 + 3 + 2) + 2, cout0 = 3 + 4 * ((1ll << n0) - 2);
    std::vector<std::pair<std::string, std::vector<long long>>> req;
    auto bn = [&](const std::string& p) {
        for (const char* f : {"weight", "bias", "running_mean", "running_var"}) req.push_back({p + "." + f, {FILTERS}});
    };
    req.push_back({"core.input_conv2d.weight", {FILTERS, cin0, 3, 3}});
    bn("core.batch_norm");
    int nb = 0;
    while (find(ts, "core.res_block_" + std::to_string(nb) + ".0.conv2d.weight")) nb++;
    if (nb == 0) NN_FAIL(TZ_EINVAL, "no residual blocks (core.res_block_0.0.conv2d.weight) found");
    if (2 * nb + 2 > conv::MAX_LAYERS) NN_FAIL(TZ_EINVAL, "%d residual blocks: at most %d", nb, (conv::MAX_LAYERS - 2) / 2);
    for (int b = 0; b < nb; b++)
        for (int j = 0; j < 2; j++) {
            const std::string p = "core.res_block_" + std::to_string(b) + "." + std::to_string(j);
            req.push_back({p + ".conv2d.weight", {FILTERS, FILTERS, 3, 3}});
            bn(p + ".batch_norm");
        }
    req.push_back({"policy.conv2d.weight", {cout0, FILTERS, 3, 3}});
    req.push_back({"policy.conv2d.bias", {cout0}});
    for (const char* head : {"value", "ube"}) {
        req.push_back({std::string(head) + ".conv2d.weight", {1, FILTERS, 1, 1}});
        req.push_back({std::string(head) + ".conv2d.bias", {1}});
        req.push_back({std::string(head) + ".linear.weight", {1, n0 * n0}});
        req.push_back({std::string(head) + ".linear.bias", {1}});
    }
    for (const auto& r : req) {
        const HostTensor* t = find(ts, r.first);
        if (!t) NN_FAIL(TZ_EINVAL, "missing tensor %s", r.first.c_str());
        if (t->shape != r.second) NN_FAIL(TZ_EINVAL, "tensor %s has the wrong shape", r.first.c_str());
    }
    *blocks = nb;
    return TZ_OK;
}

static void bind_search(tz_handle* h);

// The network state of a handle for (board size, residual blocks): activation sets, counters, masks, both weight
// sets.  Created on first use and kept across generations; re-created only when the architecture or the debug launch
// mode changes.
static int ensure_state(tz_handle* h, int blocks) {
    const int n = h->d.n, nn = n * n;
    const int want_fused = h->dbg_per_layer ? 0 : 1;
    if (h->nn && h->nn->blocks == blocks && h->nn->max_positions == h->d.Q && h->nn->fused == want_fused &&
        h->nn->cfg_chunk_tiles == h->dbg_chunk_tiles)
        return TZ_OK;
    if (h->nn) {
        cudaDeviceSynchronize();
        nn_free(h);
    }
    NnState* s = new NnState();
    h->nn = s;
    s->n = n;
    s->blocks = blocks;
    s->in_channels = 2 * (2 * n + 3 + 2) + 2;
    s->out_channels = 3 + 4 * ((1 << n) - 2);
    s->max_positions = h->d.Q;
    make_layouts(n, blocks, &s->lay, &s->raw);
    cudaDeviceGetAttribute(&s->sm_count, cudaDevAttrMultiProcessorCount, h->device);
    auto dalloc = [&](void** p, size_t bytes) -> bool {
        if (cudaMalloc(p, bytes) != cudaSuccess) return false;
        s->allocs.push_back(*p);
        return cudaMemset(*p, 0, bytes) == cudaSuccess;
    };
    // chunking: at least `tiles` pair tiles (256 rows each) per chunk, default 150 = two per CTA pair (measured
    // plateau 144..192 on 8192 6x6 positions); 0 or the per-layer debug mode = one chunk
    {
        s->fused = want_fused;
        const int tiles = h->dbg_chunk_tiles >= 0 ? h->dbg_chunk_tiles : 150;
        s->cfg_chunk_tiles = h->dbg_chunk_tiles;
        const size_t used = (size_t)s->max_positions * nn;
        const int all_tiles = (int)((used + 2 * conv::TILE_M - 1) / (2 * conv::TILE_M));
        s->chunk_min_tiles = (!s->fused || tiles <= 0 || all_tiles < 2 * tiles) ? (1 << 28) : tiles;
        const ChunkBounds cb = chunk_bounds(s->max_positions, nn, s->chunk_min_tiles);
        s->chunk_tiles = cb.chunk_tiles;
        s->max_chunks = cb.chunks;
        s->rows_set = conv::HALO + (size_t)s->chunk_tiles * (2 * conv::TILE_M) + 2 * conv::HALO;
        // Small batches of 5x5 / 6x6 positions (the single tree of `tei`: 128 leaves): N*N does not divide the 128 rows
        // of a CTA, so positions straddle CTAs and the layers of a tile wait for their neighbours' (16 us per layer).
        // Packed rows -- 5 / 3 whole positions per CTA tile, the rest of its rows dead -- make every tile independent,
        // and the local chain of the 4x4 small batches applies (activations stay in shared memory from layer to layer).
        // Worth its 16 % / 2 % of dead tensor-core rows only while every CTA has at most one tile.
        s->pack = 0;
        if (s->fused && h->dbg_chunk_tiles < 0 && conv::TILE_M % nn != 0) {
            const int per_tile = conv::TILE_M / nn;
            const int tiles = (s->max_positions + per_tile - 1) / per_tile;
            if (tiles <= 2 * (s->sm_count / 2)) {
                s->pack = per_tile;
                const size_t rows = conv::HALO + (size_t)((tiles + 1) / 2) * (2 * conv::TILE_M) + 2 * conv::HALO;
                if (rows > s->rows_set) s->rows_set = rows;
            }
        }
    }
    // both activation buffers are one allocation
    const size_t act_bytes = 2 * s->rows_set * FILTERS * 2;
    if (dalloc((void**)&s->act_x, 2 * act_bytes)) s->act_t = s->act_x + act_bytes / 2;
    if (!s->act_x ||
        !dalloc((void**)&s->head_feat, (size_t)s->max_positions * nn * 2 * sizeof(float)) ||
        !dalloc((void**)&s->perm, (size_t)s->max_positions * h->d.M * sizeof(uint16_t)) ||
        !dalloc((void**)&s->wset[0], s->lay.total) || !dalloc((void**)&s->wset[1], s->lay.total)) {
        nn_free(h);
        NN_FAIL(TZ_ENOMEM, "cudaMalloc of the network buffers failed");
    }
    {
        // lane masks: bit i of mask[start][tap] is set when tile row i (board square (start + i) mod nn)
        // has no (dy,dx) neighbour on the board
        std::vector<uint32_t> mk((size_t)(nn + 1) * 9 * 4, 0);
        for (int start = 0; start < nn; start++)
            for (int tap = 0; tap < 9; tap++) {
                const int dy = tap / 3 - 1, dx = tap % 3 - 1;
                for (int i = 0; i < conv::TILE_M; i++) {
                    const int sq = (start + i) % nn, y = sq / n, x = sq % n;
                    const bool off = y + dy < 0 || y + dy >= n || x + dx < 0 || x + dx >= n;
                    if (off) mk[((size_t)start * 9 + tap) * 4 + i / 32] |= 1u << (i % 32);
                }
            }
        // entry nn: a packed tile (positions at rows 0, nn, 2 nn, ...; the dead rows at its end take no tap at all)
        for (int tap = 0; tap < 9; tap++) {
            const int dy = tap / 3 - 1, dx = tap % 3 - 1;
            for (int i = 0; i < conv::TILE_M; i++) {
                const int sq = i % nn, y = sq / n, x = sq % n;
                const bool off = i / nn >= conv::TILE_M / nn || y + dy < 0 || y + dy >= n || x + dx < 0 || x + dx >= n;
                if (off) mk[((size_t)nn * 9 + tap) * 4 + i / 32] |= 1u << (i % 32);
            }
        }
        if (!dalloc((void**)&s->masks, mk.size() * 4) ||
            cudaMemcpy(s->masks, mk.data(), mk.size() * 4, cudaMemcpyHostToDevice) != cudaSuccess) {
            nn_free(h);
            NN_FAIL(TZ_ENOMEM, "cudaMalloc masks");
        }
    }
    if (cudaFuncSetAttribute(conv::k_conv3x3_pair, cudaFuncAttributeMaxDynamicSharedMemorySize, conv::SMEM_BYTES) !=
        cudaSuccess) {
        nn_free(h);
        NN_FAIL(TZ_ECUDA, "cudaFuncSetAttribute(k_conv3x3_pair, %d B smem) failed", conv::SMEM_BYTES);
    }
    {
        // CTA pairs that fit on the device at once: the fused network spins on other pairs' progress, so its grid
        // must never exceed this
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(2 * (s->sm_count / 2));
        cfg.blockDim = dim3(conv::THREADS);
        cfg.dynamicSmemBytes = conv::SMEM_BYTES;
        int clusters = 0;
        if (cudaOccupancyMaxActiveClusters(&clusters, conv::k_conv3x3_pair, &cfg) == cudaSuccess && clusters > 0)
            s->max_pairs = clusters < s->sm_count / 2 ? clusters : s->sm_count / 2;
        else
            s->max_pairs = s->sm_count / 2;
        if (s->pack && (s->max_positions + s->pack - 1) / s->pack > 2 * s->max_pairs) s->pack = 0;
        s->progress_len = (size_t)s->max_chunks * s->chunk_tiles * 4 + s->max_chunks + 16 + (s->pack ? 4 * (size_t)s->max_pairs : 0);
        if (!dalloc((void**)&s->progress, s->progress_len * sizeof(unsigned))) {
            nn_free(h);
            NN_FAIL(TZ_ENOMEM, "cudaMalloc progress");
        }
    }
    bool ok = cudaStreamCreateWithFlags(&s->wstream, cudaStreamNonBlocking) == cudaSuccess;
    for (cudaEvent_t* e : {&s->ev_ready, &s->ev_swap, &s->ev_h2d})
        ok = ok && cudaEventCreateWithFlags(e, cudaEventDisableTiming) == cudaSuccess;
    for (cudaEvent_t* e : {&s->ev_gen[0], &s->ev_gen[1]}) ok = ok && cudaEventCreate(e) == cudaSuccess;
    if (!ok) {
        nn_free(h);
        NN_FAIL(TZ_ECUDA, "stream / event creation failed");
    }
    cudaDeviceSynchronize();
    return TZ_OK;
}

// Raw f32 tensors -> what the upload reads, in the order RawLayout gives (plain copies, no arithmetic).  Tensors the
// caller keeps in pinned memory (tz_host_alloc) are not copied on the host at all: the upload DMAs them from where they
// are (the caller leaves them alone until the generation is complete, tz_weight_generation); tensors in pageable memory
// go through the library's pinned staging buffer.
static bool is_pinned(const void* p) {
    cudaPointerAttributes attr;
    if (cudaPointerGetAttributes(&attr, p) != cudaSuccess) {
        cudaGetLastError();
        return false;
    }
    return attr.type == cudaMemoryTypeHost;
}

static int stage_raw(tz_handle* h, const std::vector<HostTensor>& ts) {
    NnState* s = h->nn;
    const int nn = s->n * s->n;
    if (!s->head_pin && cudaHostAlloc((void**)&s->head_pin, (2 * FILTERS + 76) * sizeof(float), cudaHostAllocDefault) != cudaSuccess)
        NN_FAIL(TZ_ENOMEM, "cudaHostAlloc failed");
    if (!s->raw_dev) {
        if (cudaMalloc((void**)&s->raw_dev, s->raw.total * sizeof(float)) != cudaSuccess)
            NN_FAIL(TZ_ENOMEM, "cudaMalloc of the raw weight staging failed");
        s->allocs.push_back(s->raw_dev);
    }
    if (s->h2d_recorded) cudaEventSynchronize(s->ev_h2d);  // the previous generation's upload has read its sources
    s->direct.clear();
    bool staging_failed = false;
    auto put = [&](size_t off, const std::string& name, size_t count) {
        const float* src = find(ts, name)->data;
        if (is_pinned(src)) {
            s->direct.push_back({off, count, src});
            return;
        }
        if (!s->raw_pin && cudaHostAlloc((void**)&s->raw_pin, s->raw.total * sizeof(float), cudaHostAllocDefault) != cudaSuccess) {
            staging_failed = true;
            return;
        }
        memcpy(s->raw_pin + off, src, count * sizeof(float));
        // adjacent staged pieces merge into one copy
        if (!s->direct.empty() && s->direct.back().src == s->raw_pin + s->direct.back().off &&
            s->direct.back().off + s->direct.back().count == off)
            s->direct.back().count += count;
        else
            s->direct.push_back({off, count, s->raw_pin + off});
    };
    for (int l = 0; l < s->lay.layers; l++) {
        const bool first = l == 0, last = l == s->lay.layers - 1;
        std::string conv_name, bn_name;
        if (first) {
            conv_name = "core.input_conv2d";
            bn_name = "core.batch_norm";
        } else if (last) {
            conv_name = "policy.conv2d";
        } else {
            const std::string p = "core.res_block_" + std::to_string((l - 1) / 2) + "." + std::to_string((l - 1) % 2);
            conv_name = p + ".conv2d";
            bn_name = p + ".batch_norm";
        }
        put(s->raw.w[l], conv_name + ".weight", (size_t)s->raw.cout[l] * s->raw.cin[l] * 9);
        if (last) {
            put(s->raw.aux[l], conv_name + ".bias", (size_t)s->raw.cout[l]);  // k_fold_bias reads cout of the 256 slots
        } else {
            put(s->raw.aux[l], bn_name + ".weight", FILTERS);
            put(s->raw.aux[l] + FILTERS, bn_name + ".bias", FILTERS);
            put(s->raw.aux[l] + 2 * FILTERS, bn_name + ".running_mean", FILTERS);
            put(s->raw.aux[l] + 3 * FILTERS, bn_name + ".running_var", FILTERS);
        }
    }
    if (staging_failed) NN_FAIL(TZ_ENOMEM, "cudaHostAlloc of the %zu MB weight staging failed", s->raw.total * 4 >> 20);
    float* hd = s->head_pin;
    memset(hd, 0, (2 * FILTERS + 76) * sizeof(float));
    memcpy(hd, find(ts, "value.conv2d.weight")->data, FILTERS * sizeof(float));
    memcpy(hd + FILTERS, find(ts, "ube.conv2d.weight")->data, FILTERS * sizeof(float));
    s->direct.push_back({s->raw.heads, (size_t)(2 * FILTERS + 76), hd});
    float* misc = hd + 2 * FILTERS;  // [2] conv biases, [2][36] linear weights, [2] linear biases
    misc[0] = find(ts, "value.conv2d.bias")->data[0];
    misc[1] = find(ts, "ube.conv2d.bias")->data[0];
    memcpy(misc + 2, find(ts, "value.linear.weight")->data, nn * sizeof(float));
    memcpy(misc + 2 + 36, find(ts, "ube.linear.weight")->data, nn * sizeof(float));
    misc[2 + 72] = find(ts, "value.linear.bias")->data[0];
    misc[2 + 73] = find(ts, "ube.linear.bias")->data[0];
    return TZ_OK;
}

// wstream: wait until nobody reads `target` any more, upload the staged raw tensors, fold them into it
static int upload_and_fold(tz_handle* h, int target) {
    NnState* s = h->nn;
    if (s->swap_recorded && cudaStreamWaitEvent(s->wstream, s->ev_swap, 0) != cudaSuccess) NN_FAIL(TZ_ECUDA, "cudaStreamWaitEvent");
    cudaEventRecord(s->ev_gen[0], s->wstream);
    for (const NnState::DirectCopy& c : s->direct)
        if (cudaMemcpyAsync(s->raw_dev + c.off, c.src, c.count * sizeof(float), cudaMemcpyHostToDevice, s->wstream) != cudaSuccess)
            NN_FAIL(TZ_ECUDA, "weight upload failed");
    cudaEventRecord(s->ev_h2d, s->wstream);
    s->h2d_recorded = true;
    FoldParams fp;
    memset(&fp, 0, sizeof(fp));
    fp.layers = s->lay.layers;
    fp.raw = s->raw_dev;
    fp.set = s->wset[target];
    fp.f16 = h->nn_f16;
    for (int l = 0; l < s->lay.layers; l++) {
        FoldLayer& L = fp.L[l];
        L.w = (long long)s->raw.w[l];
        L.aux = (long long)s->raw.aux[l];
        L.out_w = (long long)s->lay.w[l];
        L.out_b = (long long)s->lay.b[l];
        L.cout = s->raw.cout[l];
        L.cin = s->raw.cin[l];
        L.cin_pad = s->lay.cin_pad[l];
        L.has_bn = s->raw.has_bn[l];
    }
    const unsigned per_layer = (unsigned)(((size_t)(FILTERS / 64) * 9 * 16384 + 255) / 256);
    k_fold_weights<<<dim3(per_layer, (unsigned)s->lay.layers), 256, 0, s->wstream>>>(fp);
    k_fold_bias<<<(unsigned)s->lay.layers, FILTERS, 0, s->wstream>>>(fp);
    cudaMemcpyAsync(s->wset[target] + s->lay.head_w, s->raw_dev + s->raw.heads, (2 * FILTERS + 76) * sizeof(float),
                    cudaMemcpyDeviceToDevice, s->wstream);
    k_set_header<<<1, 1, 0, s->wstream>>>(s->wset[target], (uint32_t)s->n, (uint32_t)s->blocks, (uint32_t)h->nn_f16,
                                          s->generation + 1);
    if (cudaGetLastError() != cudaSuccess) NN_FAIL(TZ_ECUDA, "weight fold launch failed");
    return TZ_OK;
}

// The new set (weights or novelty) is complete on wstream: launches enqueued from now on wait for it
static bool search_waits_for_wstream(tz_handle* h) {
    NnState* s = h->nn;
    return cudaEventRecord(s->ev_ready, s->wstream) == cudaSuccess && cudaStreamWaitEvent(h->stream, s->ev_ready, 0) == cudaSuccess;
}
// after a swap: the event recorded on the search stream marks the end of the swapped-out set's readers, which every
// later generation waits for before it writes into an inactive set
static void record_swap(tz_handle* h) {
    NnState* s = h->nn;
    cudaEventRecord(s->ev_swap, h->stream);
    s->swap_recorded = true;
    bind_search(h);
}

// The new weight set is complete on wstream: launches enqueued from now on read it
static int publish(tz_handle* h, int target) {
    NnState* s = h->nn;
    cudaEventRecord(s->ev_gen[1], s->wstream);
    s->gen_timed = true;
    if (!search_waits_for_wstream(h)) NN_FAIL(TZ_ECUDA, "publishing the weight set failed");
    s->set_f16[target] = h->nn_f16;
    s->active = target;
    s->generation++;
    record_swap(h);
    return TZ_OK;
}

static int to_host_tensors(const char* const* names, const float* const* data, const long long* const* shapes,
                           const int* ndims, int count, std::vector<HostTensor>* ts) {
    for (int i = 0; i < count; i++) {
        HostTensor t;
        t.name = names[i];
        t.data = data[i];
        t.shape.assign(shapes[i], shapes[i] + ndims[i]);
        ts->push_back(t);
    }
    return TZ_OK;
}

// `Net::load`: a new generation from host tensors on this handle alone.  Names and shapes are checked before anything
// is touched: a reload from a bad file (the reference keeps its previous `net` when Net::load fails,
// selfplay/src/main.rs:107-119) leaves the handle usable.  Returns once the upload is enqueued; the search stream
// waits for it by itself.
int nn_set_weights(tz_handle* h, const char* const* names, const float* const* data, const long long* const* shapes,
                   const int* ndims, int count) {
    cudaSetDevice(h->device);
    std::vector<HostTensor> ts;
    to_host_tensors(names, data, shapes, ndims, count, &ts);
    int blocks = 0, rc;
    if ((rc = validate_tensors(ts, h->d.n, &blocks)) != TZ_OK) return rc;
    if ((rc = ensure_state(h, blocks)) != TZ_OK) return rc;
    if ((rc = stage_raw(h, ts)) != TZ_OK) return rc;
    const int target = h->nn->active < 0 ? 0 : h->nn->active ^ 1;
    if ((rc = upload_and_fold(h, target)) != TZ_OK) return rc;
    // the RND estimator of a 5x5 model (rnd_learning.* / rnd_target.* / min / max) rides along with the tensors
    if ((rc = rnd_set_weights(h, names, data, shapes, ndims, count)) != TZ_OK) NN_FAIL(rc, "%s", rnd_last_error());
    return publish(h, target);
}

// One generation on every rank of the handle's communicator (comm.cu): the root folds its tensors into its inactive
// set, ncclBroadcast sends the ready 16-bit set (39 MB for the 6x6 network) to the inactive set of every other rank,
// all on the weight stream beside the running search; every rank then swaps.  Ranks other than the root pass no
// tensors, only the number of residual blocks (0 = the board's default: 20 for 5x5, else 16).
int nn_broadcast_weights(tz_handle* h, const char* const* names, const float* const* data, const long long* const* shapes,
                         const int* ndims, int count, int res_blocks, int root) {
    cudaSetDevice(h->device);
    const int nranks = comm_nranks(h), rank = comm_rank(h);
    if (root < 0 || root >= nranks) NN_FAIL(TZ_EINVAL, "root %d of %d ranks", root, nranks);
    int blocks = res_blocks > 0 ? res_blocks : (h->d.n == 5 ? 20 : 16), rc;
    std::vector<HostTensor> ts;
    if (rank == root) {
        if (count <= 0) NN_FAIL(TZ_EINVAL, "the root of a weight broadcast needs the tensors");
        to_host_tensors(names, data, shapes, ndims, count, &ts);
        int found = 0;
        if ((rc = validate_tensors(ts, h->d.n, &found)) != TZ_OK) return rc;
        if (res_blocks > 0 && found != res_blocks) NN_FAIL(TZ_EINVAL, "%d residual blocks in the tensors, %d announced", found, res_blocks);
        blocks = found;
    }
    if ((rc = ensure_state(h, blocks)) != TZ_OK) return rc;
    NnState* s = h->nn;
    const int target = s->active < 0 ? 0 : s->active ^ 1;
    if (rank == root) {
        if ((rc = stage_raw(h, ts)) != TZ_OK) return rc;
        if ((rc = upload_and_fold(h, target)) != TZ_OK) return rc;
        // the root takes the RND estimator as nn_set_weights does (a model without it switches it off); it is not part
        // of the broadcast set, so the other ranks keep theirs
        if ((rc = rnd_set_weights(h, names, data, shapes, ndims, count)) != TZ_OK) NN_FAIL(rc, "%s", rnd_last_error());
    } else {
        if (s->swap_recorded && cudaStreamWaitEvent(s->wstream, s->ev_swap, 0) != cudaSuccess) NN_FAIL(TZ_ECUDA, "cudaStreamWaitEvent");
        cudaEventRecord(s->ev_gen[0], s->wstream);
    }
    if ((rc = comm_broadcast(h, s->wset[target], s->lay.total, root, s->wstream)) != TZ_OK)
        NN_FAIL(rc, "%s", comm_last_error());
    k_check_header<<<1, 1, 0, s->wstream>>>(s->wset[target], (uint32_t)s->n, (uint32_t)s->blocks, (uint32_t)h->nn_f16,
                                            h->d.status);
    return publish(h, target);
}

// device time of the last generation on the weight stream (upload + fold + broadcast), waits for it
int nn_generation_ms(tz_handle* h, double* ms, unsigned long long* generation) {
    NnState* s = h->nn;
    if (!s || !s->gen_timed) return TZ_ENOWEIGHTS;
    if (cudaEventSynchronize(s->ev_gen[1]) != cudaSuccess) return TZ_ECUDA;
    float t = 0.0f;
    if (cudaEventElapsedTime(&t, s->ev_gen[0], s->ev_gen[1]) != cudaSuccess) return TZ_ECUDA;
    *ms = (double)t;
    if (generation) *generation = s->generation;
    return TZ_OK;
}

// read back the active weight set (parity hook: folded / arranged weights against a host restatement)
int nn_debug_weight_set(tz_handle* h, unsigned char* out, size_t cap, size_t* size) {
    NnState* s = h->nn;
    if (!s || s->active < 0) return TZ_ENOWEIGHTS;
    *size = s->lay.total;
    if (!out) return TZ_OK;
    if (cap < s->lay.total) return TZ_EINVAL;
    cudaStreamSynchronize(s->wstream);
    return cudaMemcpy(out, s->wset[s->active], s->lay.total, cudaMemcpyDeviceToHost) == cudaSuccess ? TZ_OK : TZ_ECUDA;
}

// k_expand takes the heads' inputs from the device description when the agent is the device network
static void bind_search(tz_handle* h) {
    NnState* s = h->nn;
    const bool on = s && s->active >= 0 && h->agent_kind == TZ_AGENT_NETWORK;
    h->d.nn_f16 = s && s->active >= 0 ? s->set_f16[s->active] : 0;
    h->d.nn_head_feat = on ? s->head_feat : nullptr;
    h->d.nn_head_misc = on ? reinterpret_cast<const float*>(s->wset[s->active] + s->lay.head_misc) : nullptr;
    h->d.nn_novelty_set = on ? s->simhash_set : nullptr;
    h->d.nn_novelty_idx = on ? s->simhash_idx : nullptr;
    h->d.nn_rnd_unc = on ? rnd_uncertainty(h) : nullptr;
}
void nn_bind_search(tz_handle* h) { bind_search(h); }
// every collective of a handle is issued on one stream: the weight stream once a network exists
cudaStream_t nn_collective_stream(tz_handle* h) { return h->nn && h->nn->wstream ? h->nn->wstream : h->stream; }

// test hook (no GPU needed): the kernel's own work-item schedule for `count` positions, and the bounds the host
// sizes the activation sets and progress counters with.  out[0..4] = items, chunks, chunk_tiles, chunk_rows of the
// schedule; out[4..7] = host bounds: chunks, chunk_tiles, rows per activation set; triples (chunk, layer, pair tile)
// of up to `cap` items go to out_items.
int nn_debug_schedule(int count, int count_max, int n, int chunk_min_tiles, int layers, long long* out, int* out_items,
                      int cap) {
    const int nn = n * n;
    conv::Schedule sc;
    sc.init(count, nn, chunk_min_tiles, layers);
    out[0] = sc.items;
    out[1] = sc.rows_used > 0 ? (sc.rows_used + sc.chunk_rows - 1) / sc.chunk_rows : 0;
    out[2] = sc.chunk_tiles;
    out[3] = sc.chunk_rows;
    const ChunkBounds cb = chunk_bounds(count_max, nn, chunk_min_tiles);
    out[4] = cb.chunks;
    out[5] = cb.chunk_tiles;
    out[6] = conv::HALO + (long long)cb.chunk_tiles * (2 * conv::TILE_M) + 2 * conv::HALO;
    for (int i = 0; i < sc.items && i < cap; i++) {
        const conv::Item it = sc.at(i);
        out_items[3 * i] = it.chunk;
        out_items[3 * i + 1] = it.layer;
        out_items[3 * i + 2] = it.pt;
    }
    return 0;
}

void nn_set_layer_limit(tz_handle* h, int limit) {
    if (h->nn) h->nn->layer_limit = limit;
}

// ---- forward ---------------------------------------------------------------------------------------------

// where the first and the last convolution meet the search: the queued positions and their legal-move tables
struct Boundary {
    const TzState* states;      // [count] positions (pad1[0] = white - black top flats)
    const uint16_t* actions;    // [count][M]
    const uint32_t* ranges;     // [count][36]
    const uint16_t* perm;       // [count][M] or null
    float* logits;              // [count][M]
};

static conv::Layer conv_layer(const NnState* s, int set, int l, const __nv_bfloat16* in, const __nv_bfloat16* residual,
                              __nv_bfloat16* out_act, int relu) {
    conv::Layer L;
    memset(&L, 0, sizeof(L));
    L.in = in;
    L.w = reinterpret_cast<const __nv_bfloat16*>(s->wset[set] + s->lay.w[l]);
    L.bias = reinterpret_cast<const float*>(s->wset[set] + s->lay.b[l]);
    L.residual = residual;
    L.out_act = out_act;
    L.cin = s->lay.cin_pad[l];
    L.relu = relu;
    return L;
}

// Launches p.layers[0..n_layers) as ONE persistent kernel over activation sets of `rows_set` rows holding
// one chunk (at least `chunk_min_tiles` pair tiles) each.  With more than one layer the CTA pairs synchronise through s->progress
// inside the kernel, so the launch is cooperative (all pairs resident, or it fails loudly).
static cudaError_t launch_layers(tz_handle* h, conv::Params& p, int set, const int* count_ptr, int count_max, size_t rows_set,
                                 int chunk_min_tiles, int pack = 0) {
    const NnState* s = h->nn;
    p.pack = pack;
    // what the kernel's schedule counts: positions of N*N rows, or (packed) CTA tiles of 128 rows
    const int nn = pack ? conv::TILE_M : s->n * s->n;
    const int units_max = pack ? (count_max + pack - 1) / pack : count_max;
    p.rows_set = (long long)rows_set;
    p.set_stride = (long long)rows_set * FILTERS;
    p.chunk_min_tiles = chunk_min_tiles;
    p.count_ptr = count_ptr;
    p.count_max = count_max;
    p.n = s->n;
    p.guard = conv::HALO;
    p.masks = s->masks;
    p.f16 = s->set_f16[set];
    // upper bounds of what the kernel derives from the device-side count (conv::Schedule::init)
    const int all_tiles = (units_max * nn + 2 * conv::TILE_M - 1) / (2 * conv::TILE_M);
    const ChunkBounds cb = chunk_bounds(units_max, nn, chunk_min_tiles);
    const int chunks = cb.chunks, chunk_tiles = cb.chunk_tiles;
    const size_t counters = (size_t)chunks * chunk_tiles * 4 + chunks;  // 4 channel blocks per tile, then the chunks
    p.progress = s->progress;
    p.chunk_done = s->progress + (size_t)chunks * chunk_tiles * 4;
    p.status = h->d.status;
    p.debug_drop_progress = h->dbg_drop_progress;  // watchdog test only (tz_debug_network_mode)
    const long long items = (long long)all_tiles * p.n_layers;
    const int pairs = items < s->max_pairs ? (items > 0 ? (int)items : 1) : s->max_pairs;
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(2 * pairs);
    cfg.blockDim = dim3(conv::THREADS);
    cfg.dynamicSmemBytes = conv::SMEM_BYTES;
    cfg.stream = h->stream;
    cudaLaunchAttribute attr[1];
    if (p.n_layers > 1) {
        if (counters > s->progress_len || (chunks > 1 && (size_t)chunk_tiles * 2 * conv::TILE_M + 3 * conv::HALO > rows_set))
            return cudaErrorInvalidValue;
        cudaError_t e = cudaMemsetAsync(s->progress, 0, counters * sizeof(unsigned), h->stream);
        if (e != cudaSuccess) return e;
        attr[0].id = cudaLaunchAttributeCooperative;
        attr[0].val.cooperative = 1;
        cfg.attrs = attr;
        cfg.numAttrs = 1;
    }
    return cudaLaunchKernelEx(&cfg, conv::k_conv3x3_pair, p);
}

// The whole network body: input convolution (positions -> x, the planes are encoded by its A producer), residual
// blocks (conv(x) -> t, conv(t) + x -> x; the last one also emits the value / UBE head features), policy convolution
// (x -> the legal moves' logits).  `upto` < 0: all of it; otherwise only the first `upto` convolutions (debug hook).
// Fused: one launch, else (debug mode) one launch per layer.  Returns the number of launches, or -1 when a launch
// was refused.
static int launch_network(tz_handle* h, const Boundary& io, const int* count_ptr, int count_max, int upto) {
    NnState* s = h->nn;
    const int set = s->active;
    std::vector<conv::Layer> all;
    all.push_back(conv_layer(s, set, 0, nullptr, nullptr, s->act_x, 1));
    all.back().enc_states = io.states;
    all.back().out_is_residual = 1;
    for (int l = 0; l < 2 * s->blocks; l++) {
        all.push_back((l & 1) ? conv_layer(s, set, 1 + l, s->act_t, s->act_x, s->act_x, 1)
                              : conv_layer(s, set, 1 + l, s->act_x, nullptr, s->act_t, 1));
        all.back().out_is_residual = l & 1;  // x (the block stream) is the next block's residual, t is not
    }
    all.back().head_w = reinterpret_cast<const float*>(s->wset[set] + s->lay.head_w);
    all.back().head_out = s->head_feat;
    all.push_back(conv_layer(s, set, 1 + 2 * s->blocks, s->act_x, nullptr, nullptr, 0));
    all.back().g_out = io.logits;
    all.back().g_actions = io.actions;
    all.back().g_ranges = io.ranges;
    all.back().g_perm = io.perm;
    all.back().g_stride = h->d.M;
    if (upto >= 0 && (size_t)upto < all.size()) all.resize((size_t)upto);
    int launches = 0;
    for (size_t first = 0; first < all.size();) {
        const size_t chunk = s->fused ? all.size() - first : 1;
        conv::Params p;
        for (size_t i = 0; i < chunk; i++) {
            p.layers[i] = all[first + i];
            p.dead_after[i] = nullptr;
        }
        if (chunk == all.size() && upto < 0) {
            // last reads: the block middle t by the second convolution of every block (the next block overwrites it), the
            // stream x by the policy convolution
            for (size_t i = 2; i + 1 < chunk; i += 2) p.dead_after[i] = s->act_t;
            p.dead_after[chunk - 1] = s->act_x;
        }
        p.n_layers = (int)chunk;
        p.allow_local = upto < 0;  // the debug read-backs look at the activation buffers in global memory
        const int pack = p.allow_local && chunk == all.size() ? s->pack : 0;
        if (launch_layers(h, p, set, count_ptr, count_max, s->rows_set, s->chunk_min_tiles, pack) != cudaSuccess) return -1;
        first += chunk;
        launches++;
    }
    return launches;
}

static void launch_novelty(tz_handle* h, const TzState* states, const int* count_ptr, int count_max) {
    NnState* s = h->nn;
    const TzDev& d = h->d;
    const int wblocks = (count_max + WPB - 1) / WPB;
    if (!s->simhash_set) return;
    if (s->novelty == 2)
        k_lcghash<<<wblocks, 32 * WPB, 0, h->stream>>>(states, count_ptr, count_max, d.n, d.half_komi, s->lcghash_init,
                                                       s->simhash_idx);
    else
        k_simhash<<<wblocks, 32 * WPB, 0, h->stream>>>(states, count_ptr, count_max, d.n, d.half_komi, s->simhash_matrix,
                                                       s->simhash_idx);
    h->launches += 1;
}

// The search's leaf queue (k_select filled positions, moves and per-square ranges): ONE launch; the legal logits land
// in d.logits, the head features in head_feat where k_expand finishes them.
int nn_forward_queue(tz_handle* h) {
    NnState* s = h->nn;
    if (!s || s->active < 0) return TZ_ENOWEIGHTS;
    const TzDev& d = h->d;
    const Boundary io = {d.leaf_state, d.actions, d.sq_ranges, nullptr, d.logits};
    {
        // input, tower and policy convolutions are one launch, so the sampled profile books all of it here
        ProfScope ps(h, TZ_PROF_CONV_TOWER);
        const int launched = launch_network(h, io, d.nn_count, d.Q, -1);
        if (launched < 0) {
            cudaGetLastError();
            return TZ_ECUDA;
        }
        h->launches += launched;
    }
    launch_novelty(h, d.leaf_state, d.nn_count, d.Q);
    if (rnd_forward(h, d.leaf_state, d.nn_count, d.Q) != TZ_OK) return TZ_ECUDA;
    return cudaGetLastError() == cudaSuccess ? TZ_OK : TZ_ECUDA;
}

// `impl Agent for Net`::policy_value_uncertainty for positions / action lists that came from the host (already in
// d.leaf_state / d.actions / d.n_actions): group the lists by square, run the network, finish the heads into
// d.value / d.variance.
int nn_forward_host(tz_handle* h, int count) {
    NnState* s = h->nn;
    if (!s || s->active < 0) return TZ_ENOWEIGHTS;
    if (count > s->max_positions) return TZ_EINVAL;
    const TzDev& d = h->d;
    const int wblocks = (count + WPB - 1) / WPB;
    const int limit = s->layer_limit;
    // the debug read-back shows one chunk: refuse more positions than run as a single chunk
    if (limit >= 0 && (count * d.n * d.n + 2 * conv::TILE_M - 1) / (2 * conv::TILE_M) >= 2LL * s->chunk_min_tiles)
        return TZ_EINVAL;
    cudaMemsetAsync(d.logits, 0, (size_t)count * d.M * sizeof(float), h->stream);
    k_prepare_eval<<<wblocks, 32 * WPB, 0, h->stream>>>(d.leaf_state, count, d.n, d.half_komi, s->set_f16[s->active], d.actions,
                                                        d.n_actions, d.M, d.sq_ranges, s->perm);
    const Boundary io = {d.leaf_state, d.actions, d.sq_ranges, s->perm, d.logits};
    const int launched = launch_network(h, io, nullptr, count, limit);
    if (launched < 0) {
        cudaGetLastError();
        return TZ_ECUDA;
    }
    h->launches += 1 + launched;
    if (limit >= 0) return cudaGetLastError() == cudaSuccess ? TZ_OK : TZ_ECUDA;
    launch_novelty(h, d.leaf_state, nullptr, count);
    if (rnd_forward(h, d.leaf_state, nullptr, count) != TZ_OK) return TZ_ECUDA;
    k_heads<<<wblocks, 32 * WPB, 0, h->stream>>>(s->head_feat, reinterpret_cast<const float*>(s->wset[s->active] + s->lay.head_misc),
                                                 count, d.n, s->simhash_set, s->simhash_idx, rnd_uncertainty(h), d.value, d.variance);
    h->launches += 1;
    return cudaGetLastError() == cudaSuccess ? TZ_OK : TZ_ECUDA;
}

int nn_encode_planes(tz_handle* h, const TzState* states, int count, float* out_f32) {
    const TzDev& d = h->d;
    k_encode<<<(count + WPB - 1) / WPB, 32 * WPB, 0, h->stream>>>(states, count, d.n, d.half_komi, out_f32);
    return cudaGetLastError() == cudaSuccess ? TZ_OK : TZ_ECUDA;
}

// debug read-back: which = 0 act_x, 1 act_t of the last tz_evaluate; f32 [count][n*n][256]
__global__ void k_unpad(const __nv_bfloat16* buf, int channels, int count, int n, int guard, long long rows, int f16,
                        float* out) {
    const size_t idx = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int nn = n * n;
    if (idx >= (size_t)count * nn * channels) return;
    const int c = (int)(idx % channels);
    const size_t cell = idx / channels;  // position * nn + square
    const size_t at = ((size_t)(c >> 3) * (size_t)rows + (size_t)guard + cell) * 8 + (c & 7);
    out[idx] = f16 ? __half2float(reinterpret_cast<const __half*>(buf)[at]) : __bfloat162float(buf[at]);
}

// which = 2: the 16-bit input planes as the first convolution's A producer encodes them (from the positions of the
// last tz_evaluate), f32 [count][n*n][64]
int nn_debug_read(tz_handle* h, int which, int count, float* out_dev) {
    NnState* s = h->nn;
    if (!s || s->active < 0) return TZ_ENOWEIGHTS;
    const int f16 = s->set_f16[s->active];
    if (which == 2) {
        const int cells = count * s->n * s->n;
        k_encode16<<<(cells + 127) / 128, 128, 0, h->stream>>>(h->d.leaf_state, count, s->n, f16, out_dev);
        return cudaGetLastError() == cudaSuccess ? TZ_OK : TZ_ECUDA;
    }
    const __nv_bfloat16* buf = which == 0 ? s->act_x : s->act_t;
    // the activation sets hold one chunk
    if ((count * s->n * s->n + 2 * conv::TILE_M - 1) / (2 * conv::TILE_M) >= 2LL * s->chunk_min_tiles) return TZ_EINVAL;
    const size_t total = (size_t)count * s->n * s->n * FILTERS;
    k_unpad<<<(unsigned)((total + 255) / 256), 256, 0, h->stream>>>(buf, FILTERS, count, s->n, conv::HALO,
                                                                    (long long)s->rows_set, f16, out_dev);
    return cudaGetLastError() == cudaSuccess ? TZ_OK : TZ_ECUDA;
}

// test / tuning hook: time `reps` repetitions of one residual block (2 tower convolutions) over `count` positions
// with CUDA events; returns the mean milliseconds per convolution launch.  The block stream X comes from the input
// convolution over whatever positions the last tz_evaluate left in the queue -- realistic activations, which matters
// under the power cap -- and is only read afterwards (the second convolution writes to a scratch buffer).
int nn_time_tower(tz_handle* h, int count, int reps, double* ms_per_conv) {
    NnState* s = h->nn;
    if (!s || s->active < 0) return TZ_ENOWEIGHTS;
    if (count <= 0 || count > s->max_positions || reps <= 0) return TZ_EINVAL;
    const int set = s->active;
    const size_t rows = conv::HALO + (((size_t)s->max_positions * s->n * s->n + 2 * conv::TILE_M - 1) / (2 * conv::TILE_M)) *
                                         (2 * conv::TILE_M) + 2 * conv::HALO;
    for (int i = 0; i < 3; i++)
        if (!s->tune_buf[i]) {
            if (cudaMalloc((void**)&s->tune_buf[i], rows * FILTERS * 2) != cudaSuccess) return TZ_ENOMEM;
            s->allocs.push_back(s->tune_buf[i]);
            cudaMemset(s->tune_buf[i], 0, rows * FILTERS * 2);
        }
    __nv_bfloat16 *x = s->tune_buf[0], *t = s->tune_buf[1], *scratch = s->tune_buf[2];
    auto one = [&](const conv::Layer& L) {
        conv::Params p;
        p.layers[0] = L;
        p.dead_after[0] = nullptr;
        p.n_layers = 1;
        p.allow_local = 0;
        return launch_layers(h, p, set, nullptr, count, rows, 1 << 28);
    };
    conv::Layer first = conv_layer(s, set, 0, nullptr, nullptr, x, 1);
    first.enc_states = h->d.leaf_state;
    one(first);
    const conv::Layer c1 = conv_layer(s, set, 1, x, nullptr, t, 1);
    const conv::Layer c2 = conv_layer(s, set, 2, t, x, scratch, 1);
    cudaEvent_t a, b;
    cudaEventCreate(&a);
    cudaEventCreate(&b);
    for (int i = 0; i < 2; i++) {
        one(c1);
        one(c2);
    }
    cudaEventRecord(a, h->stream);
    for (int i = 0; i < reps; i++) {
        one(c1);
        one(c2);
    }
    cudaEventRecord(b, h->stream);
    cudaEventSynchronize(b);
    float ms = 0.0f;
    cudaEventElapsedTime(&ms, a, b);
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    *ms_per_conv = (double)ms / (2.0 * reps);
    return cudaGetLastError() == cudaSuccess ? TZ_OK : TZ_ECUDA;
}

// SimHash matrix ([C*N*N][32] f32) and the optional 2^32-bit set (512 MiB, the reference's bitvec.bin)
int nn_set_simhash(tz_handle* h, const float* matrix, const unsigned char* bitset) {
    NnState* s = h->nn;
    if (!s || s->active < 0) return TZ_ENOWEIGHTS;
    cudaStreamSynchronize(h->stream);
    const size_t rows = (size_t)s->in_channels * s->n * s->n;
    if (!s->simhash_matrix) {
        if (cudaMalloc((void**)&s->simhash_matrix, rows * 32 * 4) != cudaSuccess) return TZ_ENOMEM;
        s->allocs.push_back(s->simhash_matrix);
    }
    if (!s->simhash_idx) {
        if (cudaMalloc((void**)&s->simhash_idx, (size_t)s->max_positions * 4) != cudaSuccess) return TZ_ENOMEM;
        s->allocs.push_back(s->simhash_idx);
    }
    if (cudaMemcpy(s->simhash_matrix, matrix, rows * 32 * 4, cudaMemcpyHostToDevice) != cudaSuccess) return TZ_ECUDA;
    s->novelty = 1;
    if (bitset) {
        const size_t bytes = (size_t)1 << 29;
        if (!s->simhash_set_alloc) {
            if (cudaMalloc((void**)&s->simhash_set_alloc, bytes) != cudaSuccess) return TZ_ENOMEM;
            s->allocs.push_back(s->simhash_set_alloc);
        }
        if (cudaMemcpy(s->simhash_set_alloc, bitset, bytes, cudaMemcpyHostToDevice) != cudaSuccess) return TZ_ECUDA;
        s->simhash_set = s->simhash_set_alloc;
    } else {
        s->simhash_set = nullptr;  // empty set: local uncertainty is MAXIMUM_VARIANCE everywhere
    }
    bind_search(h);
    return TZ_OK;
}

// LCG-hash novelty (net4_lcghash.rs): the per-cell multipliers and the optional 2^32-bit set; replaces SimHash
int nn_set_lcghash(tz_handle* h, const float* init, const unsigned char* bitset) {
    NnState* s = h->nn;
    if (!s || s->active < 0) return TZ_ENOWEIGHTS;
    cudaStreamSynchronize(h->stream);
    const size_t cells = (size_t)s->in_channels * s->n * s->n;
    if (!s->lcghash_init) {
        if (cudaMalloc((void**)&s->lcghash_init, cells * 4) != cudaSuccess) return TZ_ENOMEM;
        s->allocs.push_back(s->lcghash_init);
    }
    if (!s->simhash_idx) {
        if (cudaMalloc((void**)&s->simhash_idx, (size_t)s->max_positions * 4) != cudaSuccess) return TZ_ENOMEM;
        s->allocs.push_back(s->simhash_idx);
    }
    if (cudaMemcpy(s->lcghash_init, init, cells * 4, cudaMemcpyHostToDevice) != cudaSuccess) return TZ_ECUDA;
    s->novelty = 2;
    if (bitset) {
        const size_t bytes = (size_t)1 << 29;
        if (!s->simhash_set_alloc) {
            if (cudaMalloc((void**)&s->simhash_set_alloc, bytes) != cudaSuccess) return TZ_ENOMEM;
            s->allocs.push_back(s->simhash_set_alloc);
        }
        if (cudaMemcpy(s->simhash_set_alloc, bitset, bytes, cudaMemcpyHostToDevice) != cudaSuccess) return TZ_ECUDA;
        s->simhash_set = s->simhash_set_alloc;
    } else {
        s->simhash_set = nullptr;
    }
    bind_search(h);
    return TZ_OK;
}

int nn_lcghash_indices(tz_handle* h, const TzState* states, int count, uint32_t* out_dev) {
    NnState* s = h->nn;
    if (!s || !s->lcghash_init) return TZ_ENOWEIGHTS;
    k_lcghash<<<(count + WPB - 1) / WPB, 32 * WPB, 0, h->stream>>>(states, nullptr, count, h->d.n, h->d.half_komi,
                                                                   s->lcghash_init, out_dev);
    return cudaGetLastError() == cudaSuccess ? TZ_OK : TZ_ECUDA;
}

int nn_simhash_indices(tz_handle* h, const TzState* states, int count, uint32_t* out_dev) {
    NnState* s = h->nn;
    if (!s || !s->simhash_matrix) return TZ_ENOWEIGHTS;
    k_simhash<<<(count + WPB - 1) / WPB, 32 * WPB, 0, h->stream>>>(states, nullptr, count, h->d.n, h->d.half_komi,
                                                                   s->simhash_matrix, out_dev);
    return cudaGetLastError() == cudaSuccess ? TZ_OK : TZ_ECUDA;
}

// `update_counts` (net6_simhash.rs:236-241, net4_lcghash.rs `update_counts`): mark the hash index of every given
// position as seen.  The set is created (empty) on first use; indices come from the handle's current hash.
__global__ void k_set_bits(const uint32_t* __restrict__ idx, int count, uint32_t* __restrict__ set) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < count) atomicOr(&set[idx[i] >> 5], 1u << (idx[i] & 31));
}

// the empty set of a fresh network becomes a real, zeroed one before it is marked
static int ensure_marked_set(tz_handle* h) {
    NnState* s = h->nn;
    if (!s->simhash_set_alloc) {
        if (cudaMalloc((void**)&s->simhash_set_alloc, NOVELTY_BYTES) != cudaSuccess) return TZ_ENOMEM;
        s->allocs.push_back(s->simhash_set_alloc);
    }
    if (!s->simhash_set) {
        if (cudaMemsetAsync(s->simhash_set_alloc, 0, NOVELTY_BYTES, h->stream) != cudaSuccess) return TZ_ECUDA;
        s->simhash_set = s->simhash_set_alloc;
        bind_search(h);
    }
    return TZ_OK;
}

int nn_hash_kind(const tz_handle* h) { return h->nn ? h->nn->novelty : 0; }

int nn_update_counts(tz_handle* h, const TzState* states_dev, int count, uint32_t* idx_dev) {
    NnState* s = h->nn;
    if (!s || s->novelty == 0) return TZ_ENOWEIGHTS;
    if (const int erc = ensure_marked_set(h)) return erc;
    const int rc = s->novelty == 2 ? nn_lcghash_indices(h, states_dev, count, idx_dev)
                                   : nn_simhash_indices(h, states_dev, count, idx_dev);
    if (rc) return rc;
    k_set_bits<<<(count + 255) / 256, 256, 0, h->stream>>>(idx_dev, count, s->simhash_set);
    return cudaGetLastError() == cudaSuccess ? TZ_OK : TZ_ECUDA;
}

// the set as the reference saves it (bitvec.bin, 2^29 bytes); all zero while the set is still the empty one
int nn_read_novelty_set(tz_handle* h, unsigned char* out_host) {
    NnState* s = h->nn;
    if (!s || s->novelty == 0) return TZ_ENOWEIGHTS;
    const size_t bytes = (size_t)1 << 29;
    if (cudaStreamSynchronize(h->stream) != cudaSuccess) return TZ_ECUDA;
    if (!s->simhash_set) {
        memset(out_host, 0, bytes);
        return TZ_OK;
    }
    return cudaMemcpy(out_host, s->simhash_set, bytes, cudaMemcpyDeviceToHost) == cudaSuccess ? TZ_OK : TZ_ECUDA;
}

// tz_update_counts_buffer: mark the examples of a training batch (k_mark_batch) on the search stream
int nn_update_counts_buffer(tz_handle* h, const TzTargetRing& R, int batch, const unsigned long long* indices,
                            const int* symmetry, int augment, unsigned long long seed, unsigned long long size,
                            unsigned long long first) {
    NnState* s = h->nn;
    if (!s || s->novelty == 0) return TZ_ENOWEIGHTS;
    if (const int rc = ensure_marked_set(h)) return rc;
    const float* w = s->novelty == 2 ? s->lcghash_init : s->simhash_matrix;
    k_mark_batch<<<(batch + WPB - 1) / WPB, 32 * WPB, 0, h->stream>>>(R, h->d.n, h->d.half_komi, batch, indices, symmetry,
                                                                      augment, seed, size, first, s->novelty, w,
                                                                      s->simhash_set);
    h->launches += 1;
    return cudaGetLastError() == cudaSuccess ? TZ_OK : TZ_ECUDA;
}

// ---- novelty-set generations (tz_broadcast_novelty_set) ------------------------------------------------------

__global__ void k_novelty_header(uint32_t* hdr, uint32_t kind, uint32_t n) {
    hdr[0] = NOVELTY_MAGIC;
    hdr[1] = kind;
    hdr[2] = n;
    hdr[3] = 0;
}

// after a broadcast: the set that arrived must be indexed by this rank's hash (kind and board size); hdr[4] says
// whether it is not
__global__ void k_check_novelty(uint32_t* hdr, uint32_t kind, uint32_t n, uint32_t* status) {
    const bool bad = hdr[0] != NOVELTY_MAGIC || hdr[1] != kind || hdr[2] != n;
    hdr[4] = bad ? 1u : 0u;
    if (bad) atomicOr(status, TZ_ERR_WEIGHTS_MISMATCH);
}

// a rank whose check failed keeps its old set: the received one is overwritten with it (zeroes for the empty set)
// before the swap; nothing to do otherwise
__global__ void k_keep_novelty(const uint32_t* hdr, uint4* dst, const uint4* src, size_t count) {
    if (!hdr[4]) return;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x)
        dst[i] = src ? src[i] : make_uint4(0u, 0u, 0u, 0u);
}

// One set generation on every rank of the handle's communicator, on the weight stream beside the search: the root
// writes the new set into its inactive set (from a host image, or bitset = NULL: its own current set, marks enqueued
// before the call included), ncclBroadcast sends the hash kind and the set into every other rank's inactive set, and
// every rank swaps for the launches it enqueues afterwards.  The inactive set is written only after the readers of the
// last swap (ev_swap), as for the weights.
int nn_broadcast_novelty_set(tz_handle* h, const unsigned char* bitset, int root) {
    cudaSetDevice(h->device);
    const int nranks = comm_nranks(h), rank = comm_rank(h);
    if (root < 0 || root >= nranks) NN_FAIL(TZ_EINVAL, "root %d of %d ranks", root, nranks);
    if (rank != root && bitset) NN_FAIL(TZ_EINVAL, "rank %d is not the root (%d): only the root passes a set", rank, root);
    NnState* s = h->nn;
    if (!s || s->active < 0) NN_FAIL(TZ_ENOWEIGHTS, "no network: tz_set_weights / tz_broadcast_weights first");
    if (rank == root && s->novelty == 0) NN_FAIL(TZ_ENOWEIGHTS, "the root has no hash: tz_set_simhash / tz_set_lcghash first");
    if (!s->set_spare) {
        if (cudaMalloc((void**)&s->set_spare, NOVELTY_BYTES) != cudaSuccess) {
            cudaGetLastError();
            NN_FAIL(TZ_ENOMEM, "cudaMalloc of the second 512 MiB novelty set failed");
        }
        s->allocs.push_back(s->set_spare);
    }
    if (!s->set_hdr) {
        if (cudaMalloc((void**)&s->set_hdr, 8 * sizeof(uint32_t)) != cudaSuccess) NN_FAIL(TZ_ENOMEM, "cudaMalloc failed");
        s->allocs.push_back(s->set_hdr);
    }
    if (!s->ev_marks) {
        bool ok = true;
        for (cudaEvent_t* e : {&s->ev_marks, &s->ev_stage[0], &s->ev_stage[1]})
            ok = ok && cudaEventCreateWithFlags(e, cudaEventDisableTiming) == cudaSuccess;
        if (!ok) NN_FAIL(TZ_ECUDA, "event creation failed");
    }
    uint32_t* target = s->set_spare;
    if (s->swap_recorded && cudaStreamWaitEvent(s->wstream, s->ev_swap, 0) != cudaSuccess) NN_FAIL(TZ_ECUDA, "cudaStreamWaitEvent");
    if (cudaEventRecord(s->ev_marks, h->stream) != cudaSuccess) NN_FAIL(TZ_ECUDA, "cudaEventRecord");
    cudaError_t e = cudaSuccess;
    if (rank == root) {
        if (!bitset) {
            // the root's own set, once the marks enqueued before this call have landed
            e = cudaStreamWaitEvent(s->wstream, s->ev_marks, 0);
            if (e == cudaSuccess)
                e = s->simhash_set ? cudaMemcpyAsync(target, s->simhash_set, NOVELTY_BYTES, cudaMemcpyDeviceToDevice, s->wstream)
                                   : cudaMemsetAsync(target, 0, NOVELTY_BYTES, s->wstream);
        } else if (is_pinned(bitset)) {
            e = cudaMemcpyAsync(target, bitset, NOVELTY_BYTES, cudaMemcpyHostToDevice, s->wstream);
        } else {
            // pageable: through two pinned chunks in turn, so that the caller's image has been read when the call returns
            if (!s->set_pin && cudaHostAlloc((void**)&s->set_pin, 2 * NOVELTY_STAGE_BYTES, cudaHostAllocDefault) != cudaSuccess) {
                cudaGetLastError();
                s->set_pin = nullptr;
                NN_FAIL(TZ_ENOMEM, "cudaHostAlloc of the %zu MiB set staging failed", 2 * NOVELTY_STAGE_BYTES >> 20);
            }
            for (size_t off = 0, i = 0; off < NOVELTY_BYTES && e == cudaSuccess; off += NOVELTY_STAGE_BYTES, i++) {
                const int k = (int)(i & 1);
                unsigned char* pin = s->set_pin + k * NOVELTY_STAGE_BYTES;
                if (s->stage_used[k] && (e = cudaEventSynchronize(s->ev_stage[k])) != cudaSuccess) break;
                memcpy(pin, bitset + off, NOVELTY_STAGE_BYTES);
                e = cudaMemcpyAsync(reinterpret_cast<unsigned char*>(target) + off, pin, NOVELTY_STAGE_BYTES,
                                    cudaMemcpyHostToDevice, s->wstream);
                if (e == cudaSuccess) e = cudaEventRecord(s->ev_stage[k], s->wstream);
                s->stage_used[k] = true;
            }
        }
        if (e == cudaSuccess) k_novelty_header<<<1, 1, 0, s->wstream>>>(s->set_hdr, (uint32_t)s->novelty, (uint32_t)s->n);
    }
    if (e != cudaSuccess) NN_FAIL(TZ_ECUDA, "set upload failed: %s", cudaGetErrorString(e));
    int rc;
    if ((rc = comm_broadcast(h, s->set_hdr, 4 * sizeof(uint32_t), root, s->wstream)) != TZ_OK ||
        (rc = comm_broadcast(h, target, NOVELTY_BYTES, root, s->wstream)) != TZ_OK)
        NN_FAIL(rc, "%s", comm_last_error());
    if (rank != root) {
        k_check_novelty<<<1, 1, 0, s->wstream>>>(s->set_hdr, (uint32_t)s->novelty, (uint32_t)s->n, h->d.status);
        if (s->novelty) {
            // the old set as it stands after the marks enqueued before this call
            cudaStreamWaitEvent(s->wstream, s->ev_marks, 0);
            k_keep_novelty<<<4 * s->sm_count, 256, 0, s->wstream>>>(s->set_hdr, reinterpret_cast<uint4*>(target),
                                                                    reinterpret_cast<const uint4*>(s->simhash_set),
                                                                    NOVELTY_BYTES / sizeof(uint4));
        }
    }
    if (cudaGetLastError() != cudaSuccess) NN_FAIL(TZ_ECUDA, "set generation launch failed");
    if (!search_waits_for_wstream(h)) NN_FAIL(TZ_ECUDA, "publishing the novelty set failed");
    // a rank without a hash keeps having none (k_check_novelty raised the mismatch)
    if (s->novelty) {
        std::swap(s->simhash_set_alloc, s->set_spare);
        s->simhash_set = s->simhash_set_alloc;
    }
    record_swap(h);
    return TZ_OK;
}
