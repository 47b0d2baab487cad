// handle.cuh -- the opaque tz_handle behind the C ABI.
#pragma once
#include <vector>

#include "../../include/takzero_b200.h"
#include "common.cuh"

struct NnState;  // nn.cu
struct TzComm;   // comm.cu
struct RndState; // rnd.cu

struct tz_handle {
    int device = 0;
    TzDev d;
    cudaStream_t stream = nullptr;
    std::vector<void*> allocs;
    // agent
    int agent_kind = 0;
    tz_agent_fn agent_fn = nullptr;
    void* agent_ctx = nullptr;
    NnState* nn = nullptr;
    int nn_f16 = 1;  // 16-bit type the next tz_set_weights converts to: 1 fp16 (default), 0 bf16
    RndState* rnd = nullptr;  // RND local-uncertainty estimator (net5), null = the model has none
    TzComm* comm = nullptr;  // NCCL communicator of this rank (tz_comm_init), null = single GPU
    unsigned long long* reduce_buf = nullptr;  // device staging of tz_allreduce_sum
    // tz_debug_network_mode (test / measurement hooks; the defaults are the product)
    int dbg_per_layer = 0;     // one launch per convolution instead of the fused launch
    int dbg_chunk_tiles = -1;  // minimum pair tiles per chunk (-1: default 150, 0: one chunk)
    int dbg_drop_progress = 0; // CTA pair 0 withholds its tiles (watchdog test)
    int dbg_tree_warps = 0;    // warps of the search-tree wavefront kernels (0: default)
    std::vector<int> tree_games;  // what d.tree_game holds (the games of the last tz_tree* call)
    // device staging of host-facing arguments / results
    float* betas = nullptr;
    float* gumbel = nullptr;
    int gumbel_stride = 0;
    uint16_t* moves = nullptr;
    int* sym = nullptr;
    int* adj = nullptr;
    uint8_t* mask = nullptr;
    int* terminal = nullptr;
    unsigned long long* randoms = nullptr;
    TzState* fin_start = nullptr;
    uint16_t* fin_replay = nullptr;
    int* fin_len = nullptr;
    int* tbl_n = nullptr;
    uint16_t* tbl_moves = nullptr;
    uint32_t *tbl_u32a = nullptr, *tbl_u32b = nullptr, *tbl_u32c = nullptr;
    float *tbl_f32a = nullptr, *tbl_f32b = nullptr, *tbl_f32c = nullptr;
    uint32_t* root_stats = nullptr;
    float* ube = nullptr;
    float* value_target = nullptr;    // [G] reanalyze value targets
    TzState* pool = nullptr;          // device-resident positions of tz_stage_positions (the replay buffer of `reanalyze`)
    size_t pool_count = 0, pool_cap = 0;
    uint32_t* pool_idx = nullptr;     // [G]
    // pinned host staging
    unsigned char* pin_small = nullptr;
    TzState* pin_states = nullptr;
    uint16_t* pin_actions = nullptr;
    int* pin_nact = nullptr;
    float* pin_logits = nullptr;
    float* pin_value = nullptr;
    float* pin_variance = nullptr;
    // resident self-play training data (tz_selfplay_record); rec.store == nullptr: recording is off
    TzRecorder rec{};
    std::vector<void*> rec_allocs;
    bool rec_stale = false;  // positions were moved or replaced since the last recording move: drop pending records
    // bookkeeping
    unsigned long long move_counter = 0;
    unsigned long long opening_counter = 0;
    unsigned long long launches = 0;  // kernels launched by this handle
    // sampled per-kernel timing (tz_profile_begin / tz_profile_end)
    int prof_every = 0;
    unsigned long long prof_tick = 0;
    bool prof_active = false;  // the current lock-step simulation is being sampled
    std::vector<cudaEvent_t> prof_events;  // pairs (start, stop)
    std::vector<int> prof_cat;
    size_t prof_used = 0;  // pairs in use
    int* prof_counts = nullptr;  // pinned: evaluation-queue length of each sampled lock-step
    int prof_locksteps = 0;
    cudaEvent_t timer_a = nullptr, timer_b = nullptr;
};

enum { TZ_PROF_SELECT = 0, TZ_PROF_ENCODE, TZ_PROF_CONV_INPUT, TZ_PROF_CONV_TOWER, TZ_PROF_CONV_POLICY,
       TZ_PROF_HEADS, TZ_PROF_EXPAND, TZ_PROF_SYNTH, TZ_PROF_CATS };
#define TZ_PROF_MAX_PAIRS 16384
#define TZ_PROF_MAX_LOCKSTEPS 1024

// bracket one kernel launch with events when the current lock-step is sampled
struct ProfScope {
    tz_handle* h;
    bool on;
    ProfScope(tz_handle* h_, int cat) : h(h_), on(false) {
        if (!h->prof_active || h->prof_used >= TZ_PROF_MAX_PAIRS) return;
        if (h->prof_events.size() < 2 * (h->prof_used + 1)) {
            cudaEvent_t a, b;
            if (cudaEventCreate(&a) != cudaSuccess || cudaEventCreate(&b) != cudaSuccess) return;
            h->prof_events.push_back(a);
            h->prof_events.push_back(b);
            h->prof_cat.push_back(cat);
        }
        h->prof_cat[h->prof_used] = cat;
        cudaEventRecord(h->prof_events[2 * h->prof_used], h->stream);
        on = true;
    }
    ~ProfScope() {
        if (!on) return;
        cudaEventRecord(h->prof_events[2 * h->prof_used + 1], h->stream);
        h->prof_used++;
    }
};
