// api.cu -- the C ABI of libtakzero_b200.so (include/takzero_b200.h): handle, device
// memory, host <-> device staging and the lock-step drivers of
// BatchedMCTS::{simulate, gumbel_sequential_halving, step, restart_terminal_envs}
// (takzero/src/search/node/batched.rs:63-409) on top of the kernels in kernels.cu / nn.cu.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "../../include/takzero_b200.h"
#include "comm.cuh"
#include "handle.cuh"
#include "kernels.cuh"
#include "nn.cuh"

static_assert(sizeof(tz_state_t) == sizeof(TzState), "ABI state layout");

static thread_local char g_err[512] = "";

static int fail(int code, const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

#define CU(call)                                                                          \
    do {                                                                                  \
        cudaError_t e_ = (call);                                                          \
        if (e_ != cudaSuccess) return fail(TZ_ECUDA, "%s: %s", #call, cudaGetErrorString(e_)); \
    } while (0)

#define CHECK_H(h)                                                    \
    do {                                                              \
        if (!(h)) return fail(TZ_EINVAL, "null handle");              \
        CU(cudaSetDevice((h)->device));                               \
    } while (0)

void tz_internal_set_error(const char* msg) { snprintf(g_err, sizeof(g_err), "%s", msg); }  // model_file.cpp

extern "C" TZ_API const char* tz_last_error(void) { return g_err; }
extern "C" TZ_API const char* tz_version(void) { return "takzero_b200 0.1 (sm_100a)"; }

extern "C" TZ_API void* tz_host_alloc(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) return nullptr;
    return p;
}
extern "C" TZ_API void tz_host_free(void* p) {
    if (p) cudaFreeHost(p);
}

template <typename T>
static cudaError_t dmalloc(tz_handle* h, T** p, size_t count) {
    void* v = nullptr;
    cudaError_t e = cudaMalloc(&v, count * sizeof(T));
    if (e == cudaSuccess) {
        h->allocs.push_back(v);
        *p = (T*)v;
    }
    return e;
}

// Host states come from outside (the reference's `Game` cannot hold an impossible position; a C struct can):
// refuse anything the device code does not expect -- stacks taller than the 64-bit colour mask, unknown piece
// types, pieces outside the board, more pieces than a player owns.  Returns the index of the first bad state or -1.
static int first_invalid_state(const tz_state_t* states, int count, int n, const uint8_t* mask = nullptr) {
    static const int STONES[7] = {0, 0, 0, 10, 15, 21, 30}, CAPS[7] = {0, 0, 0, 0, 0, 1, 1};
    const int nn = n * n;
    for (int i = 0; i < count; i++) {
        if (mask && !mask[i]) continue;
        const tz_state_t& s = states[i];
        bool ok = s.to_move <= 1 && s.stones[0] <= STONES[n] && s.stones[1] <= STONES[n] && s.caps[0] <= CAPS[n] &&
                  s.caps[1] <= CAPS[n];
        int pieces = 0;
        for (int sq = 0; sq < TZ_MAX_SQ && ok; sq++) {
            if (sq >= nn) {
                ok = s.height[sq] == 0;
            } else if (s.height[sq] > 0) {
                ok = s.height[sq] <= 64 && s.top[sq] <= 2;
                pieces += s.height[sq];
            }
        }
        if (!ok || pieces > 2 * (STONES[n] + CAPS[n])) return i;
    }
    return -1;
}
#define CHECK_STATES(states, count, mask)                                                           \
    do {                                                                                            \
        const int bad_ = first_invalid_state((states), (count), h->d.n, (mask));                     \
        if (bad_ >= 0) return fail(TZ_EINVAL, "state %d is not a possible position of this board", bad_); \
    } while (0)

static void rec_free(tz_handle* h);

static int default_stride(int n) { return n <= 3 ? 128 : n == 4 ? 256 : n == 5 ? 512 : 1024; }

extern "C" TZ_API int tz_create(const tz_config_t* cfg, tz_handle** out) {
    if (!cfg || !out) return fail(TZ_EINVAL, "null argument");
    if (cfg->board_n < 3 || cfg->board_n > 6) return fail(TZ_EINVAL, "board_n must be 3..6");
    if (cfg->n_games <= 0) return fail(TZ_EINVAL, "n_games must be positive");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(TZ_ECUDA, "no CUDA device: takzero_b200 has no CPU fallback");
    if (cfg->device < 0 || cfg->device >= ndev) return fail(TZ_EINVAL, "bad device ordinal %d", cfg->device);
    if (cfg->move_stride > TZ_MAX_MOVES) return fail(TZ_EINVAL, "move_stride > %d", TZ_MAX_MOVES);
    CU(cudaSetDevice(cfg->device));
    tz_handle* h = new tz_handle();
    // from here on a failure releases what was made so far
#define CUH(call)                                                                        \
    do {                                                                                 \
        cudaError_t e_ = (call);                                                         \
        if (e_ != cudaSuccess) {                                                         \
            const int rc_ = fail(TZ_ECUDA, "%s: %s", #call, cudaGetErrorString(e_));      \
            tz_destroy(h);                                                               \
            return rc_;                                                                  \
        }                                                                                \
    } while (0)
    h->device = cfg->device;
    h->agent_kind = TZ_AGENT_SYNTHETIC;
    TzDev& d = h->d;
    memset(&d, 0, sizeof(d));
    d.n = cfg->board_n;
    d.nn = d.n * d.n;
    d.half_komi = cfg->half_komi;
    d.rev_limit = cfg->reversible_limit > 0 ? cfg->reversible_limit : 100;
    d.G = cfg->n_games;
    d.Q = cfg->tree_batch > cfg->n_games ? cfg->tree_batch : cfg->n_games;
    d.M = cfg->move_stride > 0 ? cfg->move_stride : default_stride(d.n);
    d.game_base = cfg->game_base;
    const size_t G = (size_t)d.G, Q = (size_t)d.Q;

    uint32_t cap = cfg->arena_slots;
    if (cap == 0) {
        size_t free_b = 0, total_b = 0;
        CUH(cudaMemGetInfo(&free_b, &total_b));
        size_t c = (size_t)((double)free_b * 0.5 / ((double)G * 2.0 * 28.0));
        if (c > 262144) c = 262144;
        if (c < 4096) c = 4096;
        cap = (uint32_t)c;
    }
    d.arena.cap = cap;
    const size_t slots = G * 2 * (size_t)cap;
    cudaError_t e = cudaSuccess;
#define DM(ptr, count)                                   \
    if (e == cudaSuccess) e = dmalloc(h, &(ptr), (count))
    DM(d.arena.eval, slots);
    DM(d.arena.meta, slots);
    DM(d.arena.visits, slots);
    DM(d.arena.prob, slots);
    DM(d.arena.std_dev, slots);
    DM(d.arena.logit, slots);
    DM(d.arena.first, slots);
    DM(d.arena.half, G);
    DM(d.arena.next_slot, G);
    DM(d.env, G);
    DM(d.start_env, G);
    DM(d.replay, G * TZ_MAX_PLIES);
    DM(d.replay_len, G);
    DM(d.traj, Q * TZ_MAX_DEPTH);
    DM(d.traj_len, Q);
    DM(d.nn_queue, Q);
    DM(d.nn_count, 1);
    DM(d.leaf_state, Q);
    DM(d.actions, Q * d.M);
    DM(d.n_actions, Q);
    DM(d.sq_ranges, Q * TZ_MAX_SQ);
    DM(d.logits, Q * d.M);
    DM(d.value, Q);
    DM(d.variance, Q);
    DM(d.tree_game, G);
    DM(d.tree_fill, G);
    DM(d.tree_slot, Q);
    float* ln_table = nullptr;
    DM(ln_table, (size_t)TZ_LN_TABLE);
    DM(d.set_child, G * TZ_MAX_K);
    DM(d.set_key, G * TZ_MAX_K);
    DM(d.set_len, G);
    DM(d.counters, G * 4);
    DM(d.status, 1);
    // host-facing staging (device side)
    DM(h->betas, G);
    DM(h->gumbel, G * d.M);
    DM(h->moves, G);
    DM(h->sym, G);
    DM(h->adj, G);
    DM(h->mask, G);
    DM(h->terminal, G);
    DM(h->randoms, G);
    DM(h->fin_start, G);
    DM(h->fin_replay, G * TZ_MAX_PLIES);
    DM(h->fin_len, G);
    DM(h->tbl_n, G);
    DM(h->tbl_moves, G * d.M);
    DM(h->tbl_u32a, G * d.M);
    DM(h->tbl_u32b, G * d.M);
    DM(h->tbl_u32c, G * d.M);
    DM(h->tbl_f32a, G * d.M);
    DM(h->tbl_f32b, G * d.M);
    DM(h->tbl_f32c, G * d.M);
    DM(h->root_stats, G * 6);
    DM(h->ube, G);
    DM(h->value_target, G);
    DM(h->pool_idx, G);
    DM(h->reduce_buf, 64);
#undef DM
    if (e != cudaSuccess) {
        const int rc = fail(TZ_ENOMEM, "cudaMalloc: %s (n_games=%d arena_slots=%u)", cudaGetErrorString(e), d.G, cap);
        tz_destroy(h);
        return rc;
    }
    d.ln_table = ln_table;
    CUH(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    // exploration_rate(n) = ln((1 + n + 500) / 500) + 4 (policy.rs:140-145), evaluated with the
    // host libm like Rust's f32::ln, in the reference's operation order
    {
        std::vector<float> tab(TZ_LN_TABLE);
        for (int i = 0; i < TZ_LN_TABLE; i++) {
            volatile float x = 1.0f + (float)i;
            x = x + 500.0f;
            x = x / 500.0f;
            volatile float l = logf(x);
            tab[i] = l + 4.0f;
        }
        CUH(cudaMemcpy(ln_table, tab.data(), sizeof(float) * TZ_LN_TABLE, cudaMemcpyHostToDevice));
    }
    CUH(cudaMemsetAsync(d.arena.half, 0, G, h->stream));
    CUH(cudaMemsetAsync(d.counters, 0, G * 4 * sizeof(unsigned long long), h->stream));
    CUH(cudaMemsetAsync(d.status, 0, sizeof(uint32_t), h->stream));
    CUH(cudaMemsetAsync(d.nn_count, 0, sizeof(int), h->stream));
    CUH(cudaMemsetAsync(d.set_len, 0, G * sizeof(int), h->stream));
    CUH(cudaMemsetAsync(h->fin_len, 0, G * sizeof(int), h->stream));
    // host staging for the callback agent and small read-backs
    CUH(cudaHostAlloc((void**)&h->pin_small, 4096, cudaHostAllocDefault));
    // every game starts from a fresh default position with an empty root
    std::vector<TzState> init(G);
    memset(init.data(), 0, G * sizeof(TzState));
    const int stones = d.n == 3 ? 10 : d.n == 4 ? 15 : d.n == 5 ? 21 : 30;
    const int caps = d.n >= 5 ? 1 : 0;
    for (size_t g = 0; g < G; g++) {
        init[g].stones[0] = init[g].stones[1] = (uint8_t)stones;
        init[g].caps[0] = init[g].caps[1] = (uint8_t)caps;
    }
    CUH(cudaMemcpyAsync(h->fin_start, init.data(), G * sizeof(TzState), cudaMemcpyHostToDevice, h->stream));
    launch_set_positions(d, h->fin_start, nullptr, h->stream);
    CUH(cudaStreamSynchronize(h->stream));
    CUH(cudaGetLastError());
#undef CUH
    *out = h;
    return TZ_OK;
}

extern "C" TZ_API void tz_destroy(tz_handle* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    nn_free(h);
    comm_destroy(h);
    rec_free(h);
    for (void* p : h->allocs) cudaFree(p);
    if (h->pool) cudaFree(h->pool);
    if (h->pin_small) cudaFreeHost(h->pin_small);
    if (h->prof_counts) cudaFreeHost(h->prof_counts);
    for (cudaEvent_t e : h->prof_events) cudaEventDestroy(e);
    if (h->timer_a) cudaEventDestroy(h->timer_a);
    if (h->timer_b) cudaEventDestroy(h->timer_b);
    if (h->pin_states) cudaFreeHost(h->pin_states);
    if (h->pin_actions) cudaFreeHost(h->pin_actions);
    if (h->pin_nact) cudaFreeHost(h->pin_nact);
    if (h->pin_logits) cudaFreeHost(h->pin_logits);
    if (h->pin_value) cudaFreeHost(h->pin_value);
    if (h->pin_variance) cudaFreeHost(h->pin_variance);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

extern "C" TZ_API int tz_sync(tz_handle* h) {
    CHECK_H(h);
    CU(cudaStreamSynchronize(h->stream));
    return TZ_OK;
}

static const char* status_text(uint32_t bits, char* buf, size_t len) {
    static const char* names[] = {"arena_full", "depth",       "no_child",      "too_many_moves",  "bad_move",
                                  "nan",        "set_empty",   "replay_full",   "network_stall",   "weights_mismatch",
                                  "targets_full"};
    buf[0] = 0;
    for (int i = 0; i < 11; i++)
        if (bits & (1u << i)) {
            strncat(buf, names[i], len - strlen(buf) - 1);
            strncat(buf, " ", len - strlen(buf) - 1);
        }
    return buf;
}

// sync + sticky device status -> return code
static int finish(tz_handle* h) {
    uint32_t* bits = (uint32_t*)h->pin_small;
    CU(cudaMemcpyAsync(bits, h->d.status, sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaGetLastError());
    if (*bits) {
        char buf[160];
        return fail(TZ_ESEARCH, "device search error bits 0x%x: %s", *bits, status_text(*bits, buf, sizeof(buf)));
    }
    return TZ_OK;
}

extern "C" TZ_API int tz_status(tz_handle* h, uint32_t* out_bits) {
    CHECK_H(h);
    uint32_t* bits = (uint32_t*)h->pin_small;
    CU(cudaMemcpyAsync(bits, h->d.status, sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    if (out_bits) *out_bits = *bits;
    return TZ_OK;
}

extern "C" TZ_API int tz_clear_status(tz_handle* h) {
    CHECK_H(h);
    CU(cudaMemsetAsync(h->d.status, 0, sizeof(uint32_t), h->stream));
    return TZ_OK;
}

extern "C" TZ_API int tz_info(tz_handle* h, int* out_move_stride, uint32_t* out_arena_slots, int* out_input_channels,
                       int* out_output_channels) {
    if (!h) return fail(TZ_EINVAL, "null handle");
    const int n = h->d.n;
    if (out_move_stride) *out_move_stride = h->d.M;
    if (out_arena_slots) *out_arena_slots = h->d.arena.cap;
    if (out_input_channels) *out_input_channels = 2 * (2 * n + 3 + 2) + 2;  // repr.rs:133-139
    if (out_output_channels) *out_output_channels = 3 + 4 * ((1 << n) - 2);  // repr.rs:103-108
    return TZ_OK;
}

// ---- rules hooks ---------------------------------------------------------------------------

struct Scratch {
    std::vector<void*> ptrs;
    ~Scratch() {
        for (void* p : ptrs) cudaFree(p);
    }
    template <typename T>
    cudaError_t get(T** p, size_t count) {
        void* v = nullptr;
        cudaError_t e = cudaMalloc(&v, (count ? count : 1) * sizeof(T));
        if (e == cudaSuccess) {
            ptrs.push_back(v);
            *p = (T*)v;
        }
        return e;
    }
};

extern "C" TZ_API int tz_legal_moves(tz_handle* h, const tz_state_t* states, int count, int stride, tz_move_t* out_moves,
                              int* out_n) {
    CHECK_H(h);
    if (!states || count < 0 || stride <= 0 || !out_moves || !out_n) return fail(TZ_EINVAL, "bad argument");
    if (count > 0) CHECK_STATES(states, count, nullptr);
    if (count == 0) return TZ_OK;
    Scratch s;
    TzState* ds;
    uint16_t* dm;
    int* dn;
    CU(s.get(&ds, (size_t)count));
    CU(s.get(&dm, (size_t)count * stride));
    CU(s.get(&dn, (size_t)count));
    CU(cudaMemcpyAsync(ds, states, (size_t)count * sizeof(TzState), cudaMemcpyHostToDevice, h->stream));
    launch_rules_probe(h->d, ds, count, stride, dm, dn, nullptr, nullptr, h->stream);
    CU(cudaMemcpyAsync(out_moves, dm, (size_t)count * stride * sizeof(uint16_t), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(out_n, dn, (size_t)count * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaGetLastError());
    return TZ_OK;
}

extern "C" TZ_API int tz_result(tz_handle* h, const tz_state_t* states, int count, int* out_terminal) {
    CHECK_H(h);
    if (!states || count < 0 || !out_terminal) return fail(TZ_EINVAL, "bad argument");
    if (count > 0) CHECK_STATES(states, count, nullptr);
    if (count == 0) return TZ_OK;
    Scratch s;
    TzState* ds;
    int* dt;
    CU(s.get(&ds, (size_t)count));
    CU(s.get(&dt, (size_t)count));
    CU(cudaMemcpyAsync(ds, states, (size_t)count * sizeof(TzState), cudaMemcpyHostToDevice, h->stream));
    launch_rules_probe(h->d, ds, count, 0, nullptr, nullptr, dt, nullptr, h->stream);
    CU(cudaMemcpyAsync(out_terminal, dt, (size_t)count * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaGetLastError());
    return TZ_OK;
}

extern "C" TZ_API int tz_game_result(tz_handle* h, const tz_state_t* states, int count, int* out_result) {
    CHECK_H(h);
    if (!states || count < 0 || !out_result) return fail(TZ_EINVAL, "bad argument");
    if (count > 0) CHECK_STATES(states, count, nullptr);
    if (count == 0) return TZ_OK;
    Scratch s;
    TzState* ds;
    int* dt;
    CU(s.get(&ds, (size_t)count));
    CU(s.get(&dt, (size_t)count));
    CU(cudaMemcpyAsync(ds, states, (size_t)count * sizeof(TzState), cudaMemcpyHostToDevice, h->stream));
    launch_rules_probe(h->d, ds, count, 0, nullptr, nullptr, nullptr, dt, h->stream);
    CU(cudaMemcpyAsync(out_result, dt, (size_t)count * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaGetLastError());
    return TZ_OK;
}

extern "C" TZ_API int tz_apply(tz_handle* h, tz_state_t* states, const tz_move_t* moves, int count, int* out_ok) {
    CHECK_H(h);
    if (!states || !moves || count < 0) return fail(TZ_EINVAL, "bad argument");
    if (count > 0) CHECK_STATES(states, count, nullptr);
    if (count == 0) return TZ_OK;
    Scratch s;
    TzState* ds;
    uint16_t* dm;
    int* dk;
    CU(s.get(&ds, (size_t)count));
    CU(s.get(&dm, (size_t)count));
    CU(s.get(&dk, (size_t)count));
    CU(cudaMemcpyAsync(ds, states, (size_t)count * sizeof(TzState), cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(dm, moves, (size_t)count * sizeof(uint16_t), cudaMemcpyHostToDevice, h->stream));
    launch_apply_moves(h->d, ds, dm, count, dk, h->stream);
    CU(cudaMemcpyAsync(states, ds, (size_t)count * sizeof(TzState), cudaMemcpyDeviceToHost, h->stream));
    if (out_ok) CU(cudaMemcpyAsync(out_ok, dk, (size_t)count * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaGetLastError());
    return TZ_OK;
}

// ---- positions --------------------------------------------------------------------------------

static int upload_mask(tz_handle* h, const uint8_t* mask, const uint8_t** dmask) {
    *dmask = nullptr;
    if (mask) {
        CU(cudaMemcpyAsync(h->mask, mask, (size_t)h->d.G, cudaMemcpyHostToDevice, h->stream));
        *dmask = h->mask;
    }
    return TZ_OK;
}

extern "C" TZ_API int tz_set_positions(tz_handle* h, const tz_state_t* states, const uint8_t* mask) {
    CHECK_H(h);
    h->rec_stale = true;
    if (!states) return fail(TZ_EINVAL, "null states");
    CHECK_STATES(states, h->d.G, mask);
    const uint8_t* dmask;
    int rc = upload_mask(h, mask, &dmask);
    if (rc) return rc;
    CU(cudaMemcpyAsync(h->d.leaf_state, states, (size_t)h->d.G * sizeof(TzState), cudaMemcpyHostToDevice, h->stream));
    launch_set_positions(h->d, h->d.leaf_state, dmask, h->stream);
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaGetLastError());
    return TZ_OK;
}

extern "C" TZ_API int tz_get_positions(tz_handle* h, tz_state_t* out) {
    CHECK_H(h);
    if (!out) return fail(TZ_EINVAL, "null out");
    CU(cudaMemcpyAsync(out, h->d.env, (size_t)h->d.G * sizeof(TzState), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return TZ_OK;
}

static int upload_openings(tz_handle* h, const int* sym, const int* adj, const int** dsym, const int** dadj) {
    *dsym = *dadj = nullptr;
    if ((sym == nullptr) != (adj == nullptr)) return fail(TZ_EINVAL, "sym and adj must both be given or both NULL");
    if (sym) {
        for (int g = 0; g < h->d.G; g++)
            if (sym[g] < 0 || sym[g] > 7 || adj[g] < 0 || adj[g] > 1) return fail(TZ_EINVAL, "bad opening for game %d", g);
        CU(cudaMemcpyAsync(h->sym, sym, (size_t)h->d.G * sizeof(int), cudaMemcpyHostToDevice, h->stream));
        CU(cudaMemcpyAsync(h->adj, adj, (size_t)h->d.G * sizeof(int), cudaMemcpyHostToDevice, h->stream));
        *dsym = h->sym;
        *dadj = h->adj;
    }
    return TZ_OK;
}

extern "C" TZ_API int tz_new_openings(tz_handle* h, const uint8_t* mask, const int* sym, const int* adj, uint64_t seed) {
    CHECK_H(h);
    h->rec_stale = true;
    const uint8_t* dmask;
    const int *dsym, *dadj;
    int rc = upload_mask(h, mask, &dmask);
    if (rc) return rc;
    rc = upload_openings(h, sym, adj, &dsym, &dadj);
    if (rc) return rc;
    launch_new_openings(h->d, dmask, dsym, dadj, seed, h->opening_counter++, h->stream);
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaGetLastError());
    return TZ_OK;
}

extern "C" TZ_API int tz_random_steps(tz_handle* h, const uint8_t* mask, int steps, uint64_t seed) {
    CHECK_H(h);
    h->rec_stale = true;
    if (steps < 0) return fail(TZ_EINVAL, "steps must be >= 0");
    const uint8_t* dmask;
    int rc = upload_mask(h, mask, &dmask);
    if (rc) return rc;
    launch_random_steps(h->d, dmask, steps, seed, h->stream);
    return finish(h);
}

extern "C" TZ_API int tz_reset_roots(tz_handle* h, const uint8_t* mask) {
    CHECK_H(h);
    h->rec_stale = true;
    const uint8_t* dmask;
    int rc = upload_mask(h, mask, &dmask);
    if (rc) return rc;
    launch_reset_roots(h->d, dmask, h->stream);
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaGetLastError());
    return TZ_OK;
}

// ---- search -------------------------------------------------------------------------------------

extern "C" TZ_API int tz_set_agent(tz_handle* h, int kind, tz_agent_fn fn, void* ctx) {
    CHECK_H(h);
    if (kind == TZ_AGENT_HOST) {
        if (!fn) return fail(TZ_EINVAL, "TZ_AGENT_HOST needs a callback");
        const size_t G = (size_t)h->d.Q, M = (size_t)h->d.M;
        // each buffer on its own: a call that failed half way is completed by the next one
        if (!h->pin_states) CU(cudaHostAlloc((void**)&h->pin_states, G * sizeof(TzState), cudaHostAllocDefault));
        if (!h->pin_actions) CU(cudaHostAlloc((void**)&h->pin_actions, G * M * sizeof(uint16_t), cudaHostAllocDefault));
        if (!h->pin_nact) CU(cudaHostAlloc((void**)&h->pin_nact, G * sizeof(int), cudaHostAllocDefault));
        if (!h->pin_logits) CU(cudaHostAlloc((void**)&h->pin_logits, G * M * sizeof(float), cudaHostAllocDefault));
        if (!h->pin_value) CU(cudaHostAlloc((void**)&h->pin_value, G * sizeof(float), cudaHostAllocDefault));
        if (!h->pin_variance) CU(cudaHostAlloc((void**)&h->pin_variance, G * sizeof(float), cudaHostAllocDefault));
    } else if (kind == TZ_AGENT_NETWORK) {
        if (!nn_ready(h)) return fail(TZ_ENOWEIGHTS, "TZ_AGENT_NETWORK needs tz_set_weights first");
    } else if (kind != TZ_AGENT_SYNTHETIC) {
        return fail(TZ_EINVAL, "unknown agent kind %d", kind);
    }
    h->agent_kind = kind;
    h->agent_fn = fn;
    h->agent_ctx = ctx;
    nn_bind_search(h);  // k_expand finishes the network's heads itself when (and only when) the network is the agent
    return TZ_OK;
}

// Agent::policy_value_uncertainty over the evaluation queue -> d.logits / d.value / d.variance
static int run_agent(tz_handle* h) {
    const TzDev& d = h->d;
    if (h->agent_kind == TZ_AGENT_SYNTHETIC) {
        ProfScope ps(h, TZ_PROF_SYNTH);
        launch_agent_synth(d, h->stream);
    } else if (h->agent_kind == TZ_AGENT_NETWORK) {
        int rc = nn_forward_queue(h);
        if (rc) return fail(rc, "network forward failed: %s", cudaGetErrorString(cudaGetLastError()));
    } else {
        int* cnt = (int*)(h->pin_small + 64);
        CU(cudaMemcpyAsync(cnt, d.nn_count, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CU(cudaStreamSynchronize(h->stream));
        const size_t c = (size_t)*cnt, M = (size_t)d.M;
        if (c > 0) {
            CU(cudaMemcpyAsync(h->pin_states, d.leaf_state, c * sizeof(TzState), cudaMemcpyDeviceToHost, h->stream));
            CU(cudaMemcpyAsync(h->pin_actions, d.actions, c * M * sizeof(uint16_t), cudaMemcpyDeviceToHost, h->stream));
            CU(cudaMemcpyAsync(h->pin_nact, d.n_actions, c * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
            CU(cudaStreamSynchronize(h->stream));
            h->agent_fn(h->agent_ctx, (int)c, (const tz_state_t*)h->pin_states, h->pin_actions, h->pin_nact, d.M,
                        h->pin_logits, h->pin_value, h->pin_variance);
            CU(cudaMemcpyAsync(d.logits, h->pin_logits, c * M * sizeof(float), cudaMemcpyHostToDevice, h->stream));
            CU(cudaMemcpyAsync(d.value, h->pin_value, c * sizeof(float), cudaMemcpyHostToDevice, h->stream));
            CU(cudaMemcpyAsync(d.variance, h->pin_variance, c * sizeof(float), cudaMemcpyHostToDevice, h->stream));
        }
    }
    return TZ_OK;
}

// one lock-step simulation of all games (batched.rs:63-128 / :266-333)
static int lockstep(tz_handle* h, int phase, int halving_i, const float* dbetas) {
    const TzDev& d = h->d;
    h->prof_active = h->prof_every > 0 && (h->prof_tick++ % (unsigned long long)h->prof_every) == 0 &&
                     h->prof_locksteps < TZ_PROF_MAX_LOCKSTEPS && h->prof_used + 64 < TZ_PROF_MAX_PAIRS;
    CU(cudaMemsetAsync(d.nn_count, 0, sizeof(int), h->stream));
    {
        ProfScope ps(h, TZ_PROF_SELECT);
        launch_select(d, phase, halving_i, dbetas, h->stream);
    }
    if (h->prof_active)
        CU(cudaMemcpyAsync(h->prof_counts + h->prof_locksteps++, d.nn_count, sizeof(int), cudaMemcpyDeviceToHost,
                           h->stream));
    {
        const int rc = run_agent(h);
        if (rc) return rc;
    }
    {
        ProfScope ps(h, TZ_PROF_EXPAND);
        launch_expand(d, h->stream);
    }
    h->prof_active = false;
    h->launches += 2 + (h->agent_kind == TZ_AGENT_SYNTHETIC ? 1 : 0);  // the network counts its own launches
    return TZ_OK;
}

static int upload_betas(tz_handle* h, const float* betas, const float** dbetas) {
    *dbetas = nullptr;
    if (betas) {
        CU(cudaMemcpyAsync(h->betas, betas, (size_t)h->d.G * sizeof(float), cudaMemcpyHostToDevice, h->stream));
        *dbetas = h->betas;
    }
    return TZ_OK;
}

extern "C" TZ_API int tz_simulate(tz_handle* h, const float* betas) {
    CHECK_H(h);
    const float* dbetas;
    int rc = upload_betas(h, betas, &dbetas);
    if (rc) return rc;
    rc = lockstep(h, 0, 0, dbetas);
    if (rc) return rc;
    return finish(h);
}

static uint32_t ilog2_u32(uint32_t x) {
    uint32_t r = 0;
    while (x >>= 1) r++;
    return r;
}

// device-resident body of gumbel_sequential_halving; moves land in h->moves
int tz_search_device(tz_handle* h, const float* dbetas, int k, uint32_t budget, const float* dgumbel, int stride) {
    const TzDev& d = h->d;
    const uint32_t steps = ilog2_u32((uint32_t)k);
    int rc = lockstep(h, 0, 0, dbetas);  // batched.rs:223
    if (rc) return rc;
    launch_gumbel_init(d, k, dgumbel, stride, h->stream);
    const uint32_t visits_per_step = budget / steps;
    uint32_t visits_to_most_visited = 0;
    int remaining = k;
    for (uint32_t step = 0; step < steps; step++) {
        const uint32_t visits_per_action = visits_per_step / (uint32_t)remaining;
        for (int i = 0; i < remaining; i++)
            for (uint32_t v = 0; v < visits_per_action; v++) {
                rc = lockstep(h, 1, i, nullptr);
                if (rc) return rc;
            }
        visits_to_most_visited += visits_per_action;
        remaining /= 2;
        launch_halve(d, dbetas, (float)visits_to_most_visited, remaining, h->stream);
    }
    launch_finalize(d, h->moves, h->stream);
    h->launches += 2 + steps;
    h->move_counter++;
    return TZ_OK;
}

extern "C" TZ_API int tz_gumbel_sequential_halving(tz_handle* h, const float* betas, int sampled_actions,
                                            uint32_t search_budget, const float* gumbel, int gumbel_stride,
                                            uint64_t seed, tz_move_t* out_moves) {
    CHECK_H(h);
    // batched.rs:215-220
    if (sampled_actions <= 0 || sampled_actions > TZ_MAX_K)
        return fail(TZ_EINVAL, "At least one action must be sampled (and at most %d)", TZ_MAX_K);
    const uint32_t steps = ilog2_u32((uint32_t)sampled_actions);
    if (steps == 0 || search_budget % (steps * (uint32_t)sampled_actions) != 0)
        return fail(TZ_EINVAL, "The search budget should be a multiple of k*log2(k) for clean visits");
    if (!out_moves) return fail(TZ_EINVAL, "null out_moves");
    const float* dbetas;
    int rc = upload_betas(h, betas, &dbetas);
    if (rc) return rc;
    const TzDev& d = h->d;
    int stride = d.M;
    if (gumbel) {
        if (gumbel_stride <= 0 || gumbel_stride > d.M) return fail(TZ_EINVAL, "gumbel_stride must be 1..%d", d.M);
        stride = gumbel_stride;
        CU(cudaMemcpyAsync(h->gumbel, gumbel, (size_t)d.G * stride * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    } else {
        launch_gumbel_noise(d, h->gumbel, stride, seed, h->move_counter, h->stream);
        h->launches += 1;
    }
    h->gumbel_stride = stride;
    rc = tz_search_device(h, dbetas, sampled_actions, search_budget, h->gumbel, stride);
    if (rc) return rc;
    CU(cudaMemcpyAsync(out_moves, h->moves, (size_t)d.G * sizeof(uint16_t), cudaMemcpyDeviceToHost, h->stream));
    return finish(h);
}

extern "C" TZ_API int tz_last_gumbel(tz_handle* h, float* out, int stride) {
    CHECK_H(h);
    if (!out || stride != h->gumbel_stride) return fail(TZ_EINVAL, "stride must equal the last search's (%d)", h->gumbel_stride);
    CU(cudaMemcpyAsync(out, h->gumbel, (size_t)h->d.G * stride * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    return TZ_OK;
}

extern "C" TZ_API int tz_step(tz_handle* h, const tz_move_t* moves) {
    CHECK_H(h);
    h->rec_stale = true;
    if (!moves) return fail(TZ_EINVAL, "null moves");
    CU(cudaMemcpyAsync(h->moves, moves, (size_t)h->d.G * sizeof(uint16_t), cudaMemcpyHostToDevice, h->stream));
    launch_step(h->d, h->moves, h->stream);
    h->launches += 1;
    return finish(h);
}

extern "C" TZ_API int tz_restart_terminal(tz_handle* h, const int* sym, const int* adj, uint64_t seed, int* out_terminal) {
    CHECK_H(h);
    h->rec_stale = true;
    if (!out_terminal) return fail(TZ_EINVAL, "null out_terminal");
    const int *dsym, *dadj;
    int rc = upload_openings(h, sym, adj, &dsym, &dadj);
    if (rc) return rc;
    launch_restart(h->d, dsym, dadj, seed, h->opening_counter++, h->terminal, h->fin_start, h->fin_replay, h->fin_len,
                   h->stream);
    h->launches += 1;
    CU(cudaMemcpyAsync(out_terminal, h->terminal, (size_t)h->d.G * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    return finish(h);
}

static int read_replay(tz_handle* h, int game, const TzState* starts, const uint16_t* replays, const int* lens,
                       tz_state_t* out_start, tz_move_t* out_moves, int cap) {
    if (game < 0 || game >= h->d.G) return fail(TZ_EINVAL, "bad game index");
    int* len = (int*)(h->pin_small + 128);
    CU(cudaMemcpyAsync(len, lens + game, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    if (out_start)
        CU(cudaMemcpyAsync(out_start, starts + game, sizeof(TzState), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    const int n = *len < cap ? *len : cap;
    if (out_moves && n > 0) {
        CU(cudaMemcpyAsync(out_moves, replays + (size_t)game * TZ_MAX_PLIES, (size_t)n * sizeof(uint16_t),
                           cudaMemcpyDeviceToHost, h->stream));
        CU(cudaStreamSynchronize(h->stream));
    }
    return *len;
}

extern "C" TZ_API int tz_finished_replay(tz_handle* h, int game, tz_state_t* out_start, tz_move_t* out_moves, int cap) {
    CHECK_H(h);
    return read_replay(h, game, h->fin_start, h->fin_replay, h->fin_len, out_start, out_moves, cap);
}

extern "C" TZ_API int tz_replay(tz_handle* h, int game, tz_state_t* out_start, tz_move_t* out_moves, int cap) {
    CHECK_H(h);
    return read_replay(h, game, h->d.start_env, h->d.replay, h->d.replay_len, out_start, out_moves, cap);
}

// ---- read-backs ---------------------------------------------------------------------------------

extern "C" TZ_API int tz_root_children(tz_handle* h, int stride, int* out_n, tz_move_t* moves, uint32_t* visits,
                                uint32_t* eval_tag, uint32_t* eval_bits, float* logit, float* prob, float* std_dev) {
    CHECK_H(h);
    const TzDev& d = h->d;
    if (stride <= 0 || stride > d.M || !out_n) return fail(TZ_EINVAL, "stride must be 1..%d", d.M);
    launch_root_table(d, stride, h->tbl_n, h->tbl_moves, h->tbl_u32a, h->tbl_u32b, h->tbl_u32c, h->tbl_f32a,
                      h->tbl_f32b, h->tbl_f32c, h->stream);
    const size_t cells = (size_t)d.G * stride;
    CU(cudaMemcpyAsync(out_n, h->tbl_n, (size_t)d.G * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
#define BACK(dst, src, type) \
    if (dst) CU(cudaMemcpyAsync(dst, src, cells * sizeof(type), cudaMemcpyDeviceToHost, h->stream))
    BACK(moves, h->tbl_moves, uint16_t);
    BACK(visits, h->tbl_u32a, uint32_t);
    BACK(eval_tag, h->tbl_u32b, uint32_t);
    BACK(eval_bits, h->tbl_u32c, uint32_t);
    BACK(logit, h->tbl_f32a, float);
    BACK(prob, h->tbl_f32b, float);
    BACK(std_dev, h->tbl_f32c, float);
#undef BACK
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaGetLastError());
    return TZ_OK;
}

extern "C" TZ_API int tz_root_stats(tz_handle* h, tz_root_t* out) {
    CHECK_H(h);
    if (!out) return fail(TZ_EINVAL, "null out");
    launch_root_stats(h->d, h->root_stats, h->stream);
    CU(cudaMemcpyAsync(out, h->root_stats, (size_t)h->d.G * 6 * sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaGetLastError());
    return TZ_OK;
}

extern "C" TZ_API int tz_targets(tz_handle* h, float visitations, float beta, int stride, float* out_policy, float* out_ube,
                          int* out_n, tz_move_t* out_moves) {
    CHECK_H(h);
    const TzDev& d = h->d;
    if (stride <= 0 || stride > d.M || !out_policy || !out_ube || !out_n) return fail(TZ_EINVAL, "bad argument");
    launch_targets(d, visitations, beta, stride, h->tbl_f32a, h->ube, h->tbl_n, out_moves ? h->tbl_moves : nullptr,
                   h->stream);
    h->launches += 1;
    const size_t cells = (size_t)d.G * stride;
    CU(cudaMemcpyAsync(out_policy, h->tbl_f32a, cells * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(out_ube, h->ube, (size_t)d.G * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(out_n, h->tbl_n, (size_t)d.G * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    if (out_moves) CU(cudaMemcpyAsync(out_moves, h->tbl_moves, cells * sizeof(uint16_t), cudaMemcpyDeviceToHost, h->stream));
    return finish(h);
}

extern "C" TZ_API int tz_select_best(tz_handle* h, tz_move_t* out_moves) {
    CHECK_H(h);
    if (!out_moves) return fail(TZ_EINVAL, "null out_moves");
    launch_select_actions(h->d, 0, 0, 0.0f, nullptr, 0, 0, h->moves, h->stream);
    h->launches += 1;
    CU(cudaMemcpyAsync(out_moves, h->moves, (size_t)h->d.G * sizeof(uint16_t), cudaMemcpyDeviceToHost, h->stream));
    return finish(h);
}

extern "C" TZ_API int tz_select_selfplay(tz_handle* h, int weighted_random_plies, uint32_t threshold, float allowed_eval_drop,
                                  const uint64_t* randoms, uint64_t seed, tz_move_t* out_moves) {
    CHECK_H(h);
    if (!out_moves) return fail(TZ_EINVAL, "null out_moves");
    const unsigned long long* dr = nullptr;
    if (randoms) {
        CU(cudaMemcpyAsync(h->randoms, randoms, (size_t)h->d.G * sizeof(uint64_t), cudaMemcpyHostToDevice, h->stream));
        dr = h->randoms;
    }
    launch_select_actions(h->d, weighted_random_plies, threshold, allowed_eval_drop, dr, seed, h->move_counter, h->moves,
                          h->stream);
    h->launches += 1;
    CU(cudaMemcpyAsync(out_moves, h->moves, (size_t)h->d.G * sizeof(uint16_t), cudaMemcpyDeviceToHost, h->stream));
    return finish(h);
}

extern "C" TZ_API int tz_counters(tz_handle* h, tz_counters_t* out) {
    CHECK_H(h);
    if (!out) return fail(TZ_EINVAL, "null out");
    std::vector<unsigned long long> c((size_t)h->d.G * 4);
    CU(cudaMemcpyAsync(c.data(), h->d.counters, c.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    memset(out, 0, sizeof(*out));
    for (int g = 0; g < h->d.G; g++) {
        out->simulations += c[(size_t)g * 4 + 0];
        out->evaluations += c[(size_t)g * 4 + 1];
        out->known += c[(size_t)g * 4 + 2];
        out->expansions += c[(size_t)g * 4 + 3];
    }
    return TZ_OK;
}

// ---- network ----------------------------------------------------------------------------------------

extern "C" TZ_API int tz_set_weights(tz_handle* h, const tz_tensor_t* tensors, int count) {
    CHECK_H(h);
    if (!tensors || count <= 0) return fail(TZ_EINVAL, "no tensors");
    std::vector<const char*> names(count);
    std::vector<const float*> data(count);
    std::vector<std::vector<long long>> shapes(count);
    std::vector<const long long*> shape_ptrs(count);
    std::vector<int> ndims(count);
    for (int i = 0; i < count; i++) {
        if (!tensors[i].name || !tensors[i].data || tensors[i].ndim < 0 || tensors[i].ndim > 4)
            return fail(TZ_EINVAL, "bad tensor %d", i);
        names[i] = tensors[i].name;
        data[i] = tensors[i].data;
        for (int k = 0; k < tensors[i].ndim; k++) shapes[i].push_back((long long)tensors[i].shape[k]);
        shape_ptrs[i] = shapes[i].data();
        ndims[i] = tensors[i].ndim;
    }
    const int rc = nn_set_weights(h, names.data(), data.data(), shape_ptrs.data(), ndims.data(), count);
    if (rc) return fail(rc, "tz_set_weights: %s", nn_last_error());
    return TZ_OK;
}

// ---- multi-GPU: NCCL communicator, weight generations, counter sums (comm.cu, nn.cu) ----------------------

extern "C" TZ_API int tz_comm_unique_id(void* out_id128) {
    if (!out_id128) return fail(TZ_EINVAL, "null out");
    const int rc = comm_unique_id(out_id128);
    if (rc) return fail(rc, "tz_comm_unique_id: %s", comm_last_error());
    return TZ_OK;
}

extern "C" TZ_API int tz_comm_init(tz_handle* h, const void* id128, int nranks, int rank) {
    CHECK_H(h);
    if (nranks > 1 && !id128) return fail(TZ_EINVAL, "null id");
    const int rc = comm_init(h, id128, nranks, rank);
    if (rc) return fail(rc, "tz_comm_init: %s", comm_last_error());
    return TZ_OK;
}

extern "C" TZ_API int tz_comm_destroy(tz_handle* h) {
    CHECK_H(h);
    CU(cudaStreamSynchronize(h->stream));
    comm_destroy(h);
    return TZ_OK;
}

extern "C" TZ_API int tz_broadcast_weights(tz_handle* h, const tz_tensor_t* tensors, int count, int res_blocks, int root) {
    CHECK_H(h);
    std::vector<const char*> names;
    std::vector<const float*> data;
    std::vector<std::vector<long long>> shapes;
    std::vector<const long long*> shape_ptrs;
    std::vector<int> ndims;
    if (root < 0 || root >= comm_nranks(h)) return fail(TZ_EINVAL, "root %d is not a rank of this communicator (%d ranks)", root, comm_nranks(h));
    if (comm_rank(h) == root) {
        if (!tensors || count <= 0) return fail(TZ_EINVAL, "the root rank passes the tensors");
        names.resize(count);
        data.resize(count);
        shapes.resize(count);
        shape_ptrs.resize(count);
        ndims.resize(count);
        for (int i = 0; i < count; i++) {
            if (!tensors[i].name || !tensors[i].data || tensors[i].ndim < 0 || tensors[i].ndim > 4)
                return fail(TZ_EINVAL, "bad tensor %d", i);
            names[i] = tensors[i].name;
            data[i] = tensors[i].data;
            for (int k = 0; k < tensors[i].ndim; k++) shapes[i].push_back((long long)tensors[i].shape[k]);
            shape_ptrs[i] = shapes[i].data();
            ndims[i] = tensors[i].ndim;
        }
    } else {
        count = 0;
    }
    const int rc = nn_broadcast_weights(h, names.data(), data.data(), shape_ptrs.data(), ndims.data(), count, res_blocks, root);
    if (rc) return fail(rc, "tz_broadcast_weights: %s", nn_last_error());
    return TZ_OK;
}

extern "C" TZ_API int tz_weight_generation(tz_handle* h, uint64_t* out_generation, double* out_ms) {
    CHECK_H(h);
    double ms = 0.0;
    unsigned long long gen = 0;
    const int rc = nn_generation_ms(h, &ms, &gen);
    if (rc) return fail(rc, "no weight generation yet");
    if (out_generation) *out_generation = gen;
    if (out_ms) *out_ms = ms;
    return TZ_OK;
}

extern "C" TZ_API int tz_allreduce_sum(tz_handle* h, uint64_t* values, int count) {
    CHECK_H(h);
    if (!values || count <= 0 || count > 64) return fail(TZ_EINVAL, "count must be 1..64");
    // all collectives of a handle go out on one stream, in the order of the calls (the same on every rank)
    cudaStream_t st = nn_collective_stream(h);
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaMemcpyAsync(h->reduce_buf, values, (size_t)count * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    const int rc = comm_allreduce_sum_u64(h, h->reduce_buf, count, st);
    if (rc) return fail(rc, "tz_allreduce_sum: %s", comm_last_error());
    CU(cudaMemcpyAsync(values, h->reduce_buf, (size_t)count * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return TZ_OK;
}

extern "C" TZ_API int tz_debug_network_mode(tz_handle* h, int per_layer_launches, int chunk_min_tiles, int drop_progress) {
    if (!h) return fail(TZ_EINVAL, "null handle");
    h->dbg_per_layer = per_layer_launches != 0;
    h->dbg_chunk_tiles = chunk_min_tiles;
    h->dbg_drop_progress = drop_progress != 0;
    return TZ_OK;
}

extern "C" TZ_API int tz_debug_tree_warps(tz_handle* h, int warps) {
    if (!h) return fail(TZ_EINVAL, "null handle");
    if (warps < 0 || warps > 8) return fail(TZ_EINVAL, "warps must be 0 (default) or 1..8");
    h->dbg_tree_warps = warps;
    return TZ_OK;
}

extern "C" TZ_API int tz_debug_weight_set(tz_handle* h, uint8_t* out, size_t cap, size_t* out_size) {
    CHECK_H(h);
    if (!out_size) return fail(TZ_EINVAL, "null out_size");
    const int rc = nn_debug_weight_set(h, out, cap, out_size);
    if (rc) return fail(rc, "tz_debug_weight_set failed (weights set? cap >= size?)");
    return TZ_OK;
}

extern "C" TZ_API int tz_evaluate(tz_handle* h, const tz_state_t* states, int count, const tz_move_t* actions,
                                  const int* n_actions, int stride, float* logits, float* values, float* variances) {
    CHECK_H(h);
    const TzDev& d = h->d;
    if (!nn_ready(h)) return fail(TZ_ENOWEIGHTS, "tz_evaluate needs tz_set_weights first");
    if (!states || !actions || !n_actions || !logits || !values || !variances) return fail(TZ_EINVAL, "null argument");
    if (count > 0) CHECK_STATES(states, count, nullptr);
    if (count <= 0 || count > d.Q) return fail(TZ_EINVAL, "count must be 1..max(n_games, tree_batch)");
    if (stride != d.M) return fail(TZ_EINVAL, "stride must equal move_stride (%d)", d.M);
    for (int i = 0; i < count; i++)
        if (n_actions[i] < 0 || n_actions[i] > stride) return fail(TZ_EINVAL, "bad n_actions[%d]", i);
    const size_t c = (size_t)count;
    CU(cudaMemcpyAsync(d.leaf_state, states, c * sizeof(TzState), cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(d.actions, actions, c * d.M * sizeof(uint16_t), cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(d.n_actions, n_actions, c * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    const int rc = nn_forward_host(h, count);
    if (rc) return fail(rc, "network forward failed: %s", cudaGetErrorString(cudaGetLastError()));
    CU(cudaMemcpyAsync(logits, d.logits, c * d.M * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(values, d.value, c * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(variances, d.variance, c * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaGetLastError());
    return TZ_OK;
}

extern "C" TZ_API int tz_encode_planes(tz_handle* h, const tz_state_t* states, int count, float* out) {
    CHECK_H(h);
    if (!states || !out || count < 0) return fail(TZ_EINVAL, "bad argument");
    if (count > 0) CHECK_STATES(states, count, nullptr);
    if (count == 0) return TZ_OK;
    const int n = h->d.n, C = 2 * (2 * n + 3 + 2) + 2;
    Scratch s;
    TzState* ds;
    float* dout;
    CU(s.get(&ds, (size_t)count));
    CU(s.get(&dout, (size_t)count * C * n * n));
    CU(cudaMemcpyAsync(ds, states, (size_t)count * sizeof(TzState), cudaMemcpyHostToDevice, h->stream));
    const int rc = nn_encode_planes(h, ds, count, dout);
    if (rc) return fail(rc, "encode failed");
    CU(cudaMemcpyAsync(out, dout, (size_t)count * C * n * n * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaGetLastError());
    return TZ_OK;
}

extern "C" TZ_API int tz_debug_layer_limit(tz_handle* h, int limit) {
    CHECK_H(h);
    if (!nn_ready(h)) return fail(TZ_ENOWEIGHTS, "no weights");
    nn_set_layer_limit(h, limit);
    return TZ_OK;
}

extern "C" TZ_API int tz_debug_activations(tz_handle* h, int which, int count, float* out) {
    CHECK_H(h);
    if (!nn_ready(h)) return fail(TZ_ENOWEIGHTS, "no weights");
    if (which < 0 || which > 2 || count <= 0 || count > h->d.Q || !out) return fail(TZ_EINVAL, "bad argument");
    const int n = h->d.n, ch = which == 2 ? 64 : 256;  // 2: the 16-bit input planes of the first convolution
    const size_t total = (size_t)count * n * n * ch;
    Scratch s;
    float* dout;
    CU(s.get(&dout, total));
    const int rc = nn_debug_read(h, which, count, dout);
    if (rc) return fail(rc, "debug read failed");
    CU(cudaMemcpyAsync(out, dout, total * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaGetLastError());
    return TZ_OK;
}

// ---- device-resident self-play move and sampled kernel timing ------------------------------------------

extern "C" TZ_API int tz_selfplay_move(tz_handle* h, const tz_selfplay_t* sp) {
    CHECK_H(h);
    if (!sp) return fail(TZ_EINVAL, "null parameters");
    if (sp->sampled_actions <= 0 || sp->sampled_actions > TZ_MAX_K)
        return fail(TZ_EINVAL, "At least one action must be sampled (and at most %d)", TZ_MAX_K);
    const uint32_t steps = ilog2_u32((uint32_t)sp->sampled_actions);
    if (steps == 0 || sp->search_budget % (steps * (uint32_t)sp->sampled_actions) != 0)
        return fail(TZ_EINVAL, "The search budget should be a multiple of k*log2(k) for clean visits");
    const TzDev& d = h->d;
    const float* dbetas = nullptr;
    if (sp->beta != 0.0f) {
        // `exploration` feature of selfplay (main.rs:81-87): beta for the first half of the batch
        std::vector<float> b((size_t)d.G, 0.0f);
        for (int g = 0; g < d.G / 2; g++) b[g] = sp->beta;
        CU(cudaMemcpyAsync(h->betas, b.data(), b.size() * sizeof(float), cudaMemcpyHostToDevice, h->stream));
        CU(cudaStreamSynchronize(h->stream));
        dbetas = h->betas;
    }
    launch_gumbel_noise(d, h->gumbel, d.M, sp->seed, h->move_counter, h->stream);
    h->gumbel_stride = d.M;
    int rc = tz_search_device(h, dbetas, sp->sampled_actions, sp->search_budget, h->gumbel, d.M);
    if (rc) return rc;
    // targets of this position (selfplay/src/main.rs:243-256) stay on the device
    launch_targets(d, sp->target_visitations, sp->target_beta, d.M, h->tbl_f32a, h->ube, h->tbl_n, nullptr, h->stream);
    const bool recording = h->rec.store != nullptr;
    if (recording) {
        if (h->rec_stale) {  // the pending records describe positions that were moved or replaced since
            CU(cudaMemsetAsync(h->rec.used, 0, 3 * (size_t)d.G * sizeof(uint32_t), h->stream));
            h->rec_stale = false;
        }
        launch_record(d, h->rec, h->tbl_f32a, h->ube, h->tbl_n, d.M, h->stream);
    }
    // plies < weighted_random_plies sample proportionally to visits, the rest keep the halving winner
    launch_select_actions(d, sp->weighted_random_plies, sp->sample_threshold, sp->allowed_eval_drop, nullptr, sp->seed,
                          h->move_counter, h->tbl_moves, h->stream);
    launch_merge_moves(d, sp->weighted_random_plies, h->tbl_moves, h->moves, h->stream);
    launch_step(d, h->moves, h->stream);
    launch_restart(d, nullptr, nullptr, sp->seed, h->opening_counter++, h->terminal, h->fin_start, h->fin_replay,
                   h->fin_len, h->stream, recording ? h->rec.result : nullptr);
    h->launches += 6;
    if (recording) {
        // restart_envs_and_complete_targets (main.rs:263-329): the exploration half is the first G/2 games
        launch_emit(d, h->rec, h->terminal, h->fin_len, h->fin_start, h->fin_replay, sp->weighted_random_plies,
                    sp->beta != 0.0f ? d.G / 2 : 0, h->stream);
        h->launches += 4;
    }
    CU(cudaGetLastError());
    return TZ_OK;
}

// ---- training data of resident self-play ------------------------------------------------------------------

static void rec_free(tz_handle* h) {
    for (void* p : h->rec_allocs) cudaFree(p);
    h->rec_allocs.clear();
    memset(&h->rec, 0, sizeof(h->rec));
    h->rec_stale = false;
}

// bytes of one queued target (env, value, ube, n, policy offset, game id) / replay (start, result, terminal, length,
// move offset, game id, exploration flag)
static const size_t TZ_TARGET_BYTES = sizeof(TzState) + 4 + 4 + 4 + 8 + 4;
static const size_t TZ_REPLAY_BYTES = sizeof(TzState) + 4 + 4 + 4 + 8 + 4 + 1;

extern "C" TZ_API int tz_selfplay_record(tz_handle* h, int enable, size_t bytes_per_game, size_t output_bytes) {
    CHECK_H(h);
    CU(cudaStreamSynchronize(h->stream));
    rec_free(h);
    if (!enable) return TZ_OK;
    const size_t G = (size_t)h->d.G, M = (size_t)h->d.M;
    const size_t worst = (size_t)TZ_MAX_PLIES * (sizeof(TzRecHead) + ((6 * M + 15) & ~(size_t)15));
    size_t free_b = 0, total_b = 0;
    CU(cudaMemGetInfo(&free_b, &total_b));
    size_t bpg = bytes_per_game;
    if (bpg == 0) {  // a quarter of the free HBM, at least 64 KiB and at most the worst case, per game
        bpg = free_b / 4 / G;
        if (bpg > worst) bpg = worst;
        if (bpg < (64 << 10)) bpg = 64 << 10;
    }
    bpg &= ~(size_t)15;  // records are 16-byte aligned
    if (bpg == 0) return fail(TZ_EINVAL, "bytes_per_game must be 0 (default) or >= 16");
    size_t out = output_bytes;
    if (out == 0) {  // half of the whole store, at most an eighth of the free HBM, at least 16 MiB
        out = G * bpg / 2;
        if (out > free_b / 8) out = free_b / 8;
        if (out < (16 << 20)) out = 16 << 20;
    }
    // the queue's split: 1/16 replay records, 1/16 replay moves, the rest targets and policy entries for a mean of
    // move_stride / 4 children per target
    const size_t mean_n = M / 4 > 0 ? M / 4 : 1;
    const size_t tp = out - out / 8;
    unsigned long long cap[TZ_Q_KINDS];
    cap[TZ_Q_TARGETS] = tp / (TZ_TARGET_BYTES + 6 * mean_n);
    cap[TZ_Q_POLICY] = (tp - cap[TZ_Q_TARGETS] * TZ_TARGET_BYTES) / 6;
    cap[TZ_Q_REPLAYS] = out / 16 / TZ_REPLAY_BYTES;
    cap[TZ_Q_MOVES] = out / 16 / 2;
    for (int q = 0; q < TZ_Q_KINDS; q++)
        if (cap[q] == 0) return fail(TZ_EINVAL, "output_bytes %zu cannot hold one replay", out);
    TzRecorder& r = h->rec;
    uint32_t* cursors = nullptr;
    cudaError_t e = cudaSuccess;
#define RM(ptr, count)                                                                  \
    if (e == cudaSuccess) {                                                             \
        void* v_ = nullptr;                                                             \
        e = cudaMalloc(&v_, (size_t)(count) * sizeof(*(ptr)));                         \
        if (e == cudaSuccess) {                                                         \
            h->rec_allocs.push_back(v_);                                                \
            (ptr) = (decltype(ptr))v_;                                                  \
        }                                                                               \
    }
    RM(r.store, G * bpg);
    RM(r.rec_off, G * TZ_MAX_PLIES);
    RM(cursors, 3 * G);
    RM(r.high_water, 1);
    RM(r.fill, TZ_Q_KINDS);
    RM(r.result, G);
    RM(r.g_count, G * TZ_Q_KINDS);
    RM(r.g_base, G * TZ_Q_KINDS);
    RM(r.t_env, cap[TZ_Q_TARGETS]);
    RM(r.t_value, cap[TZ_Q_TARGETS]);
    RM(r.t_ube, cap[TZ_Q_TARGETS]);
    RM(r.t_n, cap[TZ_Q_TARGETS]);
    RM(r.t_off, cap[TZ_Q_TARGETS]);
    RM(r.t_game, cap[TZ_Q_TARGETS]);
    RM(r.p_moves, cap[TZ_Q_POLICY]);
    RM(r.p_probs, cap[TZ_Q_POLICY]);
    RM(r.r_start, cap[TZ_Q_REPLAYS]);
    RM(r.r_result, cap[TZ_Q_REPLAYS]);
    RM(r.r_terminal, cap[TZ_Q_REPLAYS]);
    RM(r.r_len, cap[TZ_Q_REPLAYS]);
    RM(r.r_off, cap[TZ_Q_REPLAYS]);
    RM(r.r_game, cap[TZ_Q_REPLAYS]);
    RM(r.r_exploration, cap[TZ_Q_REPLAYS]);
    RM(r.r_moves, cap[TZ_Q_MOVES]);
#undef RM
    if (e != cudaSuccess) {
        rec_free(h);
        return fail(TZ_ENOMEM, "cudaMalloc of the self-play record store (%zu B per game) / queue (%zu B): %s", bpg, out,
                    cudaGetErrorString(e));
    }
    r.used = cursors;
    r.count = cursors + G;
    r.full = cursors + 2 * G;
    r.bytes_per_game = bpg;
    for (int q = 0; q < TZ_Q_KINDS; q++) r.cap[q] = cap[q];
    int rc = TZ_OK;
    if (cudaMemsetAsync(cursors, 0, 3 * G * sizeof(uint32_t), h->stream) != cudaSuccess ||
        cudaMemsetAsync(r.high_water, 0, sizeof(uint32_t), h->stream) != cudaSuccess ||
        cudaMemsetAsync(r.fill, 0, TZ_Q_KINDS * sizeof(unsigned long long), h->stream) != cudaSuccess ||
        cudaStreamSynchronize(h->stream) != cudaSuccess)
        rc = fail(TZ_ECUDA, "tz_selfplay_record: %s", cudaGetErrorString(cudaGetLastError()));
    if (rc) rec_free(h);
    return rc;
}

extern "C" TZ_API int tz_selfplay_read(tz_handle* h, tz_selfplay_data_t* io) {
    CHECK_H(h);
    if (!io) return fail(TZ_EINVAL, "null io");
    const TzRecorder& r = h->rec;
    if (!r.store) return fail(TZ_EINVAL, "recording is off: tz_selfplay_record first");
    unsigned long long* fill = (unsigned long long*)(h->pin_small + 256);
    uint32_t* hw = (uint32_t*)(h->pin_small + 256 + 8 * TZ_Q_KINDS);
    uint32_t* bits = hw + 1;
    CU(cudaMemcpyAsync(fill, r.fill, TZ_Q_KINDS * sizeof(unsigned long long), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(hw, r.high_water, sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(bits, h->d.status, sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaGetLastError());
    if (*bits & ~(uint32_t)TZ_ERR_TARGETS_FULL) {
        char buf[160];
        return fail(TZ_ESEARCH, "device search error bits 0x%x: %s", *bits, status_text(*bits, buf, sizeof(buf)));
    }
    io->n_targets = (size_t)fill[TZ_Q_TARGETS];
    io->n_policy = (size_t)fill[TZ_Q_POLICY];
    io->n_replays = (size_t)fill[TZ_Q_REPLAYS];
    io->n_moves = (size_t)fill[TZ_Q_MOVES];
    io->high_water_bytes = (size_t)*hw;
    if (io->target_cap < io->n_targets || io->policy_cap < io->n_policy || io->replay_cap < io->n_replays ||
        io->move_cap < io->n_moves)
        return fail(TZ_EINVAL, "capacity too small: the queue holds %zu targets, %zu policy entries, %zu replays, %zu moves",
                    io->n_targets, io->n_policy, io->n_replays, io->n_moves);
#define OUT(dst, src, count)                                                                                    \
    if ((dst) && (count) > 0)                                                                                   \
    CU(cudaMemcpyAsync((dst), (src), (size_t)(count) * sizeof(*(dst)), cudaMemcpyDeviceToHost, h->stream))
    OUT(io->target_env, (const tz_state_t*)r.t_env, io->n_targets);
    OUT(io->target_value, r.t_value, io->n_targets);
    OUT(io->target_ube, r.t_ube, io->n_targets);
    OUT(io->target_n, r.t_n, io->n_targets);
    OUT(io->target_offset, (const uint64_t*)r.t_off, io->n_targets);
    OUT(io->target_game, r.t_game, io->n_targets);
    OUT(io->policy_moves, r.p_moves, io->n_policy);
    OUT(io->policy_probs, r.p_probs, io->n_policy);
    OUT(io->replay_start, (const tz_state_t*)r.r_start, io->n_replays);
    OUT(io->replay_result, r.r_result, io->n_replays);
    OUT(io->replay_terminal, r.r_terminal, io->n_replays);
    OUT(io->replay_length, r.r_len, io->n_replays);
    OUT(io->replay_offset, (const uint64_t*)r.r_off, io->n_replays);
    OUT(io->replay_game, r.r_game, io->n_replays);
    OUT(io->replay_exploration, r.r_exploration, io->n_replays);
    OUT(io->replay_moves, r.r_moves, io->n_moves);
#undef OUT
    CU(cudaMemsetAsync(r.fill, 0, TZ_Q_KINDS * sizeof(unsigned long long), h->stream));
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaGetLastError());
    return TZ_OK;
}

// ---- reanalyze (reanalyze/src/main.rs:147-235) without per-batch host buffers ----------------------------------------

extern "C" TZ_API int tz_stage_positions(tz_handle* h, const tz_state_t* states, size_t count) {
    CHECK_H(h);
    if (!states || count == 0) return fail(TZ_EINVAL, "no positions");
    for (size_t lo = 0; lo < count; lo += 1 << 20) {
        const int part = (int)(count - lo < (size_t)(1 << 20) ? count - lo : (size_t)(1 << 20));
        const int bad = first_invalid_state(states + lo, part, h->d.n);
        if (bad >= 0) return fail(TZ_EINVAL, "state %zu is not a possible position of this board", lo + (size_t)bad);
    }
    CU(cudaStreamSynchronize(h->stream));
    if (count > h->pool_cap) {
        if (h->pool) cudaFree(h->pool);
        h->pool = nullptr;
        h->pool_cap = 0;
        if (cudaMalloc((void**)&h->pool, count * sizeof(TzState)) != cudaSuccess)
            return fail(TZ_ENOMEM, "cudaMalloc of %zu staged positions failed", count);
        h->pool_cap = count;
    }
    CU(cudaMemcpyAsync(h->pool, states, count * sizeof(TzState), cudaMemcpyHostToDevice, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    h->pool_count = count;
    return TZ_OK;
}

// one reanalyze batch: fresh roots from staged positions, search, targets -- everything stays on the device
extern "C" TZ_API int tz_reanalyze_batch(tz_handle* h, const uint32_t* pool_indices, const tz_reanalyze_t* rp) {
    CHECK_H(h);
    if (!rp) return fail(TZ_EINVAL, "null parameters");
    if (rp->sampled_actions <= 0 || rp->sampled_actions > TZ_MAX_K)
        return fail(TZ_EINVAL, "At least one action must be sampled (and at most %d)", TZ_MAX_K);
    const uint32_t steps = ilog2_u32((uint32_t)rp->sampled_actions);
    if (steps == 0 || rp->search_budget % (steps * (uint32_t)rp->sampled_actions) != 0)
        return fail(TZ_EINVAL, "The search budget should be a multiple of k*log2(k) for clean visits");
    const TzDev& d = h->d;
    if (pool_indices) {
        if (h->pool_count == 0) return fail(TZ_EINVAL, "tz_stage_positions first");
        for (int g = 0; g < d.G; g++)
            if (pool_indices[g] >= h->pool_count) return fail(TZ_EINVAL, "pool index %u of game %d out of range", pool_indices[g], g);
        CU(cudaMemcpyAsync(h->pool_idx, pool_indices, (size_t)d.G * sizeof(uint32_t), cudaMemcpyHostToDevice, h->stream));
        launch_gather_positions(d, h->pool, h->pool_idx, h->stream);  // *node = Node::default(); *env = replay_env
        h->launches += 1;
        h->rec_stale = true;
    }
    launch_gumbel_noise(d, h->gumbel, d.M, rp->seed, h->move_counter, h->stream);
    h->gumbel_stride = d.M;
    const int rc = tz_search_device(h, nullptr, rp->sampled_actions, rp->search_budget, h->gumbel, d.M);  // ZERO_BETA
    if (rc) return rc;
    launch_targets(d, -1.0f, rp->target_beta, d.M, h->tbl_f32a, h->ube, h->tbl_n, h->tbl_moves, h->stream);
    launch_reanalyze_values(d, h->moves, h->value_target, h->stream);
    h->launches += 3;
    CU(cudaGetLastError());
    return TZ_OK;
}

// the targets of the last tz_reanalyze_batch: improved policy with most_visited_count() visitations, UBE target,
// value target, per root the child count and moves
extern "C" TZ_API int tz_reanalyze_read(tz_handle* h, int stride, float* out_policy, float* out_ube, float* out_value,
                                        int* out_n, tz_move_t* out_moves) {
    CHECK_H(h);
    const TzDev& d = h->d;
    if (stride != d.M || !out_policy || !out_ube || !out_value || !out_n || !out_moves)
        return fail(TZ_EINVAL, "stride must equal move_stride (%d) and all outputs must be given", d.M);
    const size_t cells = (size_t)d.G * stride;
    CU(cudaMemcpyAsync(out_policy, h->tbl_f32a, cells * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(out_moves, h->tbl_moves, cells * sizeof(uint16_t), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(out_ube, h->ube, (size_t)d.G * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(out_value, h->value_target, (size_t)d.G * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(out_n, h->tbl_n, (size_t)d.G * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    return finish(h);
}

extern "C" TZ_API int tz_launch_count(tz_handle* h, uint64_t* out) {
    if (!h || !out) return fail(TZ_EINVAL, "null argument");
    *out = h->launches;
    return TZ_OK;
}

extern "C" TZ_API int tz_profile_begin(tz_handle* h, int sample_every) {
    CHECK_H(h);
    if (sample_every < 0) return fail(TZ_EINVAL, "sample_every must be >= 0");
    CU(cudaStreamSynchronize(h->stream));
    if (!h->prof_counts)
        CU(cudaHostAlloc((void**)&h->prof_counts, TZ_PROF_MAX_LOCKSTEPS * sizeof(int), cudaHostAllocDefault));
    h->prof_every = sample_every;
    h->prof_tick = 0;
    h->prof_used = 0;
    h->prof_locksteps = 0;
    return TZ_OK;
}

extern "C" TZ_API int tz_profile_end(tz_handle* h, tz_profile_t* out) {
    CHECK_H(h);
    if (!out) return fail(TZ_EINVAL, "null out");
    CU(cudaStreamSynchronize(h->stream));
    memset(out, 0, sizeof(*out));
    for (size_t i = 0; i < h->prof_used; i++) {
        float ms = 0.0f;
        CU(cudaEventElapsedTime(&ms, h->prof_events[2 * i], h->prof_events[2 * i + 1]));
        const int c = h->prof_cat[i];
        out->ms[c] += ms;
        out->launches[c] += 1;
    }
    out->locksteps = (uint64_t)h->prof_locksteps;
    for (int i = 0; i < h->prof_locksteps; i++) out->positions += (uint64_t)h->prof_counts[i];
    h->prof_every = 0;
    return TZ_OK;
}

// device-side stopwatch on the library's stream (CUDA events), for callers that time whole moves
extern "C" TZ_API int tz_timer_start(tz_handle* h) {
    CHECK_H(h);
    if (!h->timer_a) {
        CU(cudaEventCreate(&h->timer_a));
        CU(cudaEventCreate(&h->timer_b));
    }
    CU(cudaEventRecord(h->timer_a, h->stream));
    return TZ_OK;
}

extern "C" TZ_API int tz_timer_stop(tz_handle* h, double* out_ms) {
    CHECK_H(h);
    if (!h->timer_a || !out_ms) return fail(TZ_EINVAL, "tz_timer_start first");
    CU(cudaEventRecord(h->timer_b, h->stream));
    CU(cudaEventSynchronize(h->timer_b));
    float ms = 0.0f;
    CU(cudaEventElapsedTime(&ms, h->timer_a, h->timer_b));
    *out_ms = (double)ms;
    return TZ_OK;
}

extern "C" TZ_API int tz_debug_time_tower(tz_handle* h, int count, int reps, double* ms_per_conv) {
    CHECK_H(h);
    if (!ms_per_conv) return fail(TZ_EINVAL, "null out");
    const int rc = nn_time_tower(h, count, reps, ms_per_conv);
    if (rc) return fail(rc, "tz_debug_time_tower failed (weights set? count <= n_games?)");
    return TZ_OK;
}

extern "C" TZ_API int tz_debug_expf(tz_handle* h, const float* in, int count, float* out) {
    CHECK_H(h);
    if (!in || !out || count < 0) return fail(TZ_EINVAL, "bad argument");
    if (count == 0) return TZ_OK;
    Scratch s;
    float *din, *dout;
    CU(s.get(&din, (size_t)count));
    CU(s.get(&dout, (size_t)count));
    CU(cudaMemcpyAsync(din, in, (size_t)count * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    launch_debug_expf(din, count, dout, h->stream);
    CU(cudaMemcpyAsync(out, dout, (size_t)count * sizeof(float), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaGetLastError());
    return TZ_OK;
}

extern "C" TZ_API int tz_debug_schedule(int count, int count_max, int board_n, int chunk_min_tiles, int layers,
                                        long long* out, int* out_items, int cap) {
    if (!out || count < 0 || count > count_max || board_n < 3 || board_n > 6 || chunk_min_tiles <= 0 || layers <= 0 ||
        (cap > 0 && !out_items))
        return fail(TZ_EINVAL, "bad argument");
    return nn_debug_schedule(count, count_max, board_n, chunk_min_tiles, layers, out, out_items, cap);
}

extern "C" TZ_API int tz_set_simhash(tz_handle* h, const float* matrix, const uint8_t* bitset) {
    CHECK_H(h);
    if (!matrix) return fail(TZ_EINVAL, "null matrix");
    CU(cudaStreamSynchronize(h->stream));
    const int rc = nn_set_simhash(h, matrix, bitset);
    if (rc) return fail(rc, "tz_set_simhash failed (tz_set_weights first; the set needs 512 MiB of HBM)");
    return TZ_OK;
}

extern "C" TZ_API int tz_simhash_indices(tz_handle* h, const tz_state_t* states, int count, uint32_t* out) {
    CHECK_H(h);
    if (!states || !out || count <= 0) return fail(TZ_EINVAL, "bad argument");
    if (count > 0) CHECK_STATES(states, count, nullptr);
    Scratch s;
    TzState* ds;
    uint32_t* dout;
    CU(s.get(&ds, (size_t)count));
    CU(s.get(&dout, (size_t)count));
    CU(cudaMemcpyAsync(ds, states, (size_t)count * sizeof(TzState), cudaMemcpyHostToDevice, h->stream));
    const int rc = nn_simhash_indices(h, ds, count, dout);
    if (rc) return fail(rc, "tz_simhash_indices needs tz_set_simhash first");
    CU(cudaMemcpyAsync(out, dout, (size_t)count * sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaGetLastError());
    return TZ_OK;
}

extern "C" TZ_API int tz_set_lcghash(tz_handle* h, const float* init, const uint8_t* bitset) {
    CHECK_H(h);
    if (!init) return fail(TZ_EINVAL, "null init");
    CU(cudaStreamSynchronize(h->stream));
    const int rc = nn_set_lcghash(h, init, bitset);
    if (rc) return fail(rc, "tz_set_lcghash failed (tz_set_weights first; the set needs 512 MiB of HBM)");
    return TZ_OK;
}

extern "C" TZ_API int tz_lcghash_indices(tz_handle* h, const tz_state_t* states, int count, uint32_t* out) {
    CHECK_H(h);
    if (!states || !out || count <= 0) return fail(TZ_EINVAL, "bad argument");
    if (count > 0) CHECK_STATES(states, count, nullptr);
    Scratch s;
    TzState* ds;
    uint32_t* dout;
    CU(s.get(&ds, (size_t)count));
    CU(s.get(&dout, (size_t)count));
    CU(cudaMemcpyAsync(ds, states, (size_t)count * sizeof(TzState), cudaMemcpyHostToDevice, h->stream));
    const int rc = nn_lcghash_indices(h, ds, count, dout);
    if (rc) return fail(rc, "tz_lcghash_indices needs tz_set_lcghash first");
    CU(cudaMemcpyAsync(out, dout, (size_t)count * sizeof(uint32_t), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaGetLastError());
    return TZ_OK;
}

extern "C" TZ_API int tz_update_counts(tz_handle* h, const tz_state_t* states, int count) {
    CHECK_H(h);
    if (!states || count <= 0) return fail(TZ_EINVAL, "bad argument");
    CHECK_STATES(states, count, nullptr);
    Scratch s;
    TzState* ds;
    uint32_t* didx;
    CU(s.get(&ds, (size_t)count));
    CU(s.get(&didx, (size_t)count));
    CU(cudaMemcpyAsync(ds, states, (size_t)count * sizeof(TzState), cudaMemcpyHostToDevice, h->stream));
    const int rc = nn_update_counts(h, ds, count, didx);
    if (rc) return fail(rc, "tz_update_counts needs tz_set_simhash / tz_set_lcghash first (the set takes 512 MiB of HBM)");
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaGetLastError());
    return TZ_OK;
}

extern "C" TZ_API int tz_read_novelty_set(tz_handle* h, uint8_t* out, size_t cap) {
    CHECK_H(h);
    if (!out || cap < ((size_t)1 << 29)) return fail(TZ_EINVAL, "out must hold 2^29 bytes");
    const int rc = nn_read_novelty_set(h, out);
    if (rc) return fail(rc, "tz_read_novelty_set needs tz_set_simhash / tz_set_lcghash first");
    return TZ_OK;
}

// ---- search trees (tei / analysis): Node::simulate_simple, simulate_batch, descend, principal_variation ----
// The trees of a call are its selected games, tree t the t-th of them in game order; one CTA (one warp for the PV) per
// tree.  The tz_tree_* calls are the same code with game 0 selected.

static std::vector<int> selected_games(const tz_handle* h, const uint8_t* mask) {
    std::vector<int> games;
    for (int g = 0; g < h->d.G; g++)
        if (!mask || mask[g]) games.push_back(g);
    return games;
}

// d.tree_game = games (copied only when it changed: the one-tree calls select game 0 every time)
static int upload_trees(tz_handle* h, const std::vector<int>& games) {
    if (games == h->tree_games) return TZ_OK;
    h->tree_games.clear();  // stays empty if the copy fails
    CU(cudaMemcpyAsync(h->d.tree_game, games.data(), games.size() * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    h->tree_games = games;
    return TZ_OK;
}

static int trees_simulate(tz_handle* h, const std::vector<int>& games, float beta, int batch_size, int max_forwards) {
    const TzDev& d = h->d;
    const int trees = (int)games.size();
    if (batch_size <= 0) return fail(TZ_EINVAL, "batch_size must be >= 1");
    if ((long long)trees * batch_size > d.Q)
        return fail(TZ_EINVAL, "selected games (%d) x batch_size (%d) must be <= max(n_games, tree_batch) (%d): raise tree_batch",
                    trees, batch_size, d.Q);
    if (trees == 0) return TZ_OK;
    h->rec_stale = true;
    int rc = upload_trees(h, games);
    if (rc) return rc;
    h->prof_active = false;
    CU(cudaMemsetAsync(d.nn_count, 0, sizeof(int), h->stream));  // the trees append their leaves
    launch_tree_forward(d, trees, beta, batch_size, max_forwards, h->dbg_tree_warps, h->stream);
    rc = run_agent(h);
    if (rc) return rc;
    launch_tree_backward(d, trees, batch_size, h->dbg_tree_warps, h->stream);
    h->launches += 2;
    return finish(h);
}

extern "C" TZ_API int tz_tree_simulate_simple(tz_handle* h, float beta) {
    CHECK_H(h);
    return trees_simulate(h, {0}, beta, 1, 1);  // mcts.rs:235-266
}

extern "C" TZ_API int tz_tree_simulate_batch(tz_handle* h, float beta, int batch_size) {
    CHECK_H(h);
    return trees_simulate(h, {0}, beta, batch_size, 4 * batch_size);  // mcts.rs:268-328
}

extern "C" TZ_API int tz_trees_simulate_batch(tz_handle* h, const uint8_t* mask, float beta, int batch_size) {
    CHECK_H(h);
    return trees_simulate(h, selected_games(h, mask), beta, batch_size, 4 * batch_size);
}

extern "C" TZ_API int tz_trees_descend(tz_handle* h, const uint8_t* mask, const tz_move_t* moves) {
    CHECK_H(h);
    if (!moves) return fail(TZ_EINVAL, "null moves");
    if (selected_games(h, mask).empty()) return TZ_OK;
    h->rec_stale = true;
    const uint8_t* dmask;
    int rc = upload_mask(h, mask, &dmask);
    if (rc) return rc;
    CU(cudaMemcpyAsync(h->moves, moves, (size_t)h->d.G * sizeof(uint16_t), cudaMemcpyHostToDevice, h->stream));
    launch_step(h->d, h->moves, h->stream, dmask);
    h->launches += 1;
    return finish(h);
}

extern "C" TZ_API int tz_tree_descend(tz_handle* h, tz_move_t move) {
    CHECK_H(h);
    std::vector<uint16_t> mv((size_t)h->d.G, 0);
    std::vector<uint8_t> mask((size_t)h->d.G, 0);
    mv[0] = move;
    mask[0] = 1;
    return tz_trees_descend(h, mask.data(), mv.data());
}

// principal variations of the trees of `games`: moves [trees][cap] (cap <= move_stride), lens [trees]
static int trees_pv(tz_handle* h, const std::vector<int>& games, int cap, std::vector<uint16_t>* moves, std::vector<int>* lens) {
    const int trees = (int)games.size();
    int rc = upload_trees(h, games);
    if (rc) return rc;
    launch_tree_pv(h->d, trees, h->tbl_moves, cap, h->tbl_n, h->stream);
    moves->resize((size_t)trees * cap);
    lens->resize(trees);
    CU(cudaMemcpyAsync(moves->data(), h->tbl_moves, moves->size() * sizeof(uint16_t), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaMemcpyAsync(lens->data(), h->tbl_n, (size_t)trees * sizeof(int), cudaMemcpyDeviceToHost, h->stream));
    CU(cudaStreamSynchronize(h->stream));
    CU(cudaGetLastError());
    return TZ_OK;
}

extern "C" TZ_API int tz_tree_principal_variation(tz_handle* h, tz_move_t* out_moves, int cap) {
    CHECK_H(h);
    if (!out_moves || cap <= 0) return fail(TZ_EINVAL, "bad argument");
    if (cap > h->d.M) cap = h->d.M;
    std::vector<uint16_t> moves;
    std::vector<int> lens;
    const int rc = trees_pv(h, {0}, cap, &moves, &lens);
    if (rc) return rc;
    std::copy(moves.begin(), moves.begin() + lens[0], out_moves);
    return lens[0];
}

extern "C" TZ_API int tz_trees_principal_variation(tz_handle* h, const uint8_t* mask, int cap, tz_move_t* out_moves,
                                                   int* out_len) {
    CHECK_H(h);
    if (!out_moves || !out_len || cap <= 0) return fail(TZ_EINVAL, "bad argument");
    const std::vector<int> games = selected_games(h, mask);
    std::fill(out_len, out_len + h->d.G, 0);
    if (games.empty()) return TZ_OK;
    const int dcap = cap < h->d.M ? cap : h->d.M;
    std::vector<uint16_t> moves;
    std::vector<int> lens;
    const int rc = trees_pv(h, games, dcap, &moves, &lens);
    if (rc) return rc;
    for (size_t t = 0; t < games.size(); t++) {
        const int g = games[t];
        std::copy(moves.begin() + t * dcap, moves.begin() + t * dcap + lens[t], out_moves + (size_t)g * cap);
        out_len[g] = lens[t];
    }
    return TZ_OK;
}

// BatchedMCTS::apply_noise (batched.rs:146-151) support: store host-computed priors / logits of the roots
extern "C" TZ_API int tz_set_root_priors(tz_handle* h, int stride, const float* prob, const float* logit) {
    CHECK_H(h);
    const TzDev& d = h->d;
    if (!prob || !logit || stride <= 0 || stride > d.M) return fail(TZ_EINVAL, "bad argument");
    const size_t cells = (size_t)d.G * stride;
    CU(cudaMemcpyAsync(h->tbl_f32a, prob, cells * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    CU(cudaMemcpyAsync(h->tbl_f32b, logit, cells * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    launch_set_root_priors(d, stride, h->tbl_f32a, h->tbl_f32b, h->stream);
    h->launches += 1;
    return finish(h);
}

extern "C" TZ_API int tz_set_network_dtype(tz_handle* h, int dtype) {
    if (!h) return fail(TZ_EINVAL, "null handle");
    if (dtype != TZ_DTYPE_BF16 && dtype != TZ_DTYPE_F16) return fail(TZ_EINVAL, "dtype must be TZ_DTYPE_BF16 or TZ_DTYPE_F16");
    h->nn_f16 = dtype == TZ_DTYPE_F16;
    return TZ_OK;
}
