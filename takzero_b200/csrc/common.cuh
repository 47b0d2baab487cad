// common.cuh -- shared constants / layouts for the takzero_b200 CUDA library (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#define TZ_MAX_SQ 36
#define TZ_MAX_MOVES 1024      // upper bound on legal moves of one position (N <= 6)
#define TZ_MAX_DEPTH 256       // longest selection path kept per game
#define TZ_MAX_K 64            // largest `sampled_actions` of sequential halving
#define TZ_MAX_PLIES 1024      // longest recorded replay
#define TZ_WARPS_PER_BLOCK 4   // warp-per-game kernels: 4 games per CTA
#define TZ_LN_TABLE (1 << 20)  // exploration_rate(n) tabulated for n < 2^20

enum { TZ_FLAT = 0, TZ_WALL = 1, TZ_CAP = 2 };
enum { TZ_E_VALUE = 0, TZ_E_WIN = 1, TZ_E_LOSS = 2, TZ_E_DRAW = 3 };
enum { TZ_T_NONE = 0, TZ_T_WIN = 1, TZ_T_LOSS = 2, TZ_T_DRAW = 3 };

// Packed game state: identical bytes on host (tz_state_t in include/takzero_b200.h)
// and device.  One 384-byte record per game, 128-byte aligned, so a warp loads a
// game with three coalesced 128-byte transactions.
struct __align__(16) TzState {
    uint64_t stack[TZ_MAX_SQ];  // bit i = colour (1 = black) of the piece at height i
    uint8_t height[TZ_MAX_SQ];
    uint8_t top[TZ_MAX_SQ];     // TZ_FLAT / TZ_WALL / TZ_CAP, valid when height > 0
    uint8_t to_move;            // 0 white, 1 black
    uint8_t stones[2];
    uint8_t caps[2];
    uint8_t pad0;
    uint16_t ply;
    uint16_t reversible_plies;
    uint8_t pad1[14];  // device copies in the evaluation queue keep derived data here (encode.cuh): pad1[0] = white -
                       // black top flats, bytes 372..383 = the position's scalar input planes as 16-bit pairs
};
static_assert(sizeof(TzState) == 384, "TzState must be 384 bytes");

// Per-game search tree: a struct-of-arrays arena of node slots (u32 / f32 per field)
//   eval      f32 bits of Value(v), or the ply of a known result
//   meta      bits 0..15 move that leads to the node, 16..17 eval tag, 18..31 child count
//   visits, prob, std_dev, logit
//   first     slot of the first child (children of one node are contiguous, in
//             `possible_moves` order); 0 = no children
// Every game owns two halves of `cap` slots; slot 0 of the active half is the root and
// children blocks are bump-allocated in expansion order.  `tz_step` re-roots by copying
// the kept subtree breadth-first into the other half (Cheney copy), which both frees the
// discarded siblings and compacts the arena.
struct TzArena {
    uint32_t* eval;
    uint32_t* meta;
    uint32_t* visits;
    float* prob;
    float* std_dev;
    float* logit;
    uint32_t* first;
    uint8_t* half;        // [G] active half
    uint32_t* next_slot;  // [G] bump pointer inside the active half
    uint32_t cap;         // slots per half
};

__host__ __device__ inline uint32_t tz_meta(uint32_t move, uint32_t tag, uint32_t nchild) {
    return (move & 0xffffu) | (tag << 16) | (nchild << 18);
}
__host__ __device__ inline uint32_t tz_meta_move(uint32_t m) { return m & 0xffffu; }
__host__ __device__ inline uint32_t tz_meta_tag(uint32_t m) { return (m >> 16) & 3u; }
__host__ __device__ inline uint32_t tz_meta_nchild(uint32_t m) { return m >> 18; }

// error bits accumulated in the handle's device-side status word
enum {
    TZ_ERR_ARENA_FULL = 1,
    TZ_ERR_DEPTH = 2,
    TZ_ERR_NO_CHILD = 4,
    TZ_ERR_TOO_MANY_MOVES = 8,
    TZ_ERR_BAD_MOVE = 16,
    TZ_ERR_NAN = 32,
    TZ_ERR_SET_EMPTY = 64,
    TZ_ERR_REPLAY_FULL = 128,
    TZ_ERR_NETWORK_STALL = 256,
    TZ_ERR_WEIGHTS_MISMATCH = 512,
    TZ_ERR_TARGETS_FULL = 1024,
};

// Device-side view of one handle, passed by value to every kernel.
struct TzDev {
    int n, nn, half_komi, rev_limit;
    int G;          // games on this device
    int Q;          // evaluation-queue capacity: max(G, tree_batch)
    int M;          // stride of per-position move / logit rows (<= TZ_MAX_MOVES)
    int game_base;  // global id of game 0 (multi-GPU sharding)
    TzArena arena;
    TzState* env;        // [G] root positions
    TzState* start_env;  // [G] position the current replay started from
    uint16_t* replay;    // [G][TZ_MAX_PLIES] moves played since start_env
    int* replay_len;     // [G]
    // one lock-step simulation
    uint32_t* traj;      // [Q][TZ_MAX_DEPTH] node slots of the selection path: by game (k_select), by queue slot (k_tree_*)
    int* traj_len;       // [Q] same index
    int* nn_queue;       // [G] evaluation-queue slot -> game
    int* nn_count;       // [1] queue length
    TzState* leaf_state; // [G] leaf positions, by queue slot
    uint16_t* actions;   // [G][M] legal moves of the leaf, by queue slot
    int* n_actions;      // [G] by queue slot
    uint32_t* sq_ranges; // [Q][36] by queue slot and square (row * N + col): index of the first legal move that starts
                         // on the square | number of such moves << 16 (moves of one square are contiguous)
    float* logits;       // [G][M] legal-move logits, by queue slot
    float* value;        // [G] by queue slot
    float* variance;     // [G] by queue slot
    // device network (nn.cu): when nn_head_feat is set, k_expand computes value / variance of queue slot q from the two
    // head features per row the last tower convolution left there, instead of reading value[] / variance[]
    int nn_f16;                      // 16-bit type of the active weight set (the queued scalar planes are stored in it)
    const float* nn_head_feat;       // [Q * N*N][2]
    const float* nn_head_misc;       // conv biases, linear weights / biases of the value and UBE heads
    const uint32_t* nn_novelty_set;  // 2^32-bit set or null (empty)
    const uint32_t* nn_novelty_idx;  // [Q] hash index of every queued position
    const float* nn_rnd_unc;         // [Q] normalized RND uncertainty of every queued position (net5), or null
    const float* ln_table;  // exploration_rate(n), n < TZ_LN_TABLE (host libm logf)
    // search trees (k_tree_*, one CTA per tree)
    int* tree_game;  // [G] game of tree t
    int* tree_fill;  // [G] leaves tree t queued in the last forward
    int* tree_slot;  // [Q] queue slot of tree t's i-th leaf (commit order) at t * batch_size + i
    // sequential halving
    uint16_t* set_child;  // [G][TZ_MAX_K] candidate set (root child index)
    float* set_key;       // [G][TZ_MAX_K] logit + gumbel
    int* set_len;         // [G]
    unsigned long long* counters;  // [G][4] simulations, evaluations, known, expansions
    uint32_t* status;              // [1] sticky error bits
};

// Training data of resident self-play (tz_selfplay_record / tz_selfplay_read).
// Pending records: every game owns `bytes_per_game` bytes of `store`; a record is a TzRecHead followed by n f32
// improved-policy probabilities and n u16 moves (child order), padded to 16 bytes.  When a game ends its records are
// completed with their value and emitted, with the game's replay, into the output queue: struct-of-arrays with one
// array per field of tz_selfplay_data_t, so that tz_selfplay_read is one copy per array.
struct __align__(16) TzRecHead {
    TzState env;  // the root position before the move
    int p;        // replay index of the move (replay_len at that moment)
    int n;        // children of the root
    float ube;    // UBE target
    int pad;
};
static_assert(sizeof(TzRecHead) == 400, "record header is 400 bytes");

enum { TZ_Q_TARGETS = 0, TZ_Q_POLICY, TZ_Q_REPLAYS, TZ_Q_MOVES, TZ_Q_KINDS };

struct TzRecorder {
    // pending records; used / count / full are one allocation [3][G] (one memset clears every cursor)
    unsigned char* store;       // [G][bytes_per_game]
    uint32_t* rec_off;          // [G][TZ_MAX_PLIES] byte offset of each record inside the game's region
    uint32_t* used;             // [G] bytes in use
    uint32_t* count;            // [G] records
    uint32_t* full;             // [G] the region ran out: no more records until the game ends
    uint32_t* high_water;       // [1] most bytes one game has used
    unsigned long long bytes_per_game;
    // output queue
    TzState* t_env;
    float* t_value;
    float* t_ube;
    int* t_n;
    unsigned long long* t_off;  // first policy entry of the target
    int* t_game;                // global game id
    uint16_t* p_moves;
    float* p_probs;
    TzState* r_start;
    int* r_result;              // tz_game_result code of the final position
    int* r_terminal;            // tz_result code of the final position (side to move)
    int* r_len;
    unsigned long long* r_off;  // first move of the replay in r_moves
    int* r_game;
    uint8_t* r_exploration;
    uint16_t* r_moves;
    unsigned long long cap[TZ_Q_KINDS];  // entries of targets, policy, replays, moves
    unsigned long long* fill;            // [TZ_Q_KINDS] entries in the queue
    // emission of one move
    int* result;                // [G] tz_game_result of every game k_restart finished
    unsigned long long* g_count;  // [G][TZ_Q_KINDS] what each finished game emits
    unsigned long long* g_base;   // [G][TZ_Q_KINDS] where it goes; g_base[g][0] = ~0 when it does not fit
};

// Target buffer (tz_target_buffer): a ring of `cap` slots with a fixed stride.  Target number k ever appended lives in
// slot k % cap; the ones kept are the last min(appended, cap).
struct TzTargetRing {
    TzState* env;      // [cap]
    float* value;      // [cap]
    float* ube;        // [cap]
    int* n;            // [cap] entries
    uint16_t* moves;   // [cap][stride]
    float* probs;      // [cap][stride]
    unsigned long long cap;
    int stride;
    unsigned long long* appended;  // [1] targets ever appended
    unsigned long long* range;     // [2] source entries [lo, hi) of the append in flight
    unsigned int* ticket;          // [1] blocks of k_target_append done (the last one advances `appended`)
};
