/*
 * takzero_b200.h -- C ABI of libtakzero_b200.so, the B200-native batched self-play search.
 *
 * The reference (ViliamVadocz/takzero, Rust) has no FFI of its own: its extension points are
 * the traits `Environment` (takzero/src/search/env.rs:11-25), `Agent` (search/agent.rs:5-14),
 * `Network` (network/mod.rs:10-45) and the struct `BatchedMCTS` (search/node/batched.rs:24-409).
 * Every entry point below names the reference item it replaces; INTEGRATION.md shows the
 * `extern "C"` block a Rust maintainer would add to bind them.
 *
 * Conventions: plain pointers and sizes only; all `host` pointers are caller-owned host
 * memory (pinned memory from tz_host_alloc makes the copies asynchronous); device memory is
 * owned by the handle.  Calls on one handle must come from one thread at a time.  Every call
 * returns 0 on success or a negative TZ_E* code, with a message in tz_last_error(); nothing
 * panics or throws across the ABI (the reference panics on the same conditions).
 * There is no CPU fallback: without a CUDA device tz_create fails.
 */
#ifndef TAKZERO_B200_H
#define TAKZERO_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define TZ_API __attribute__((visibility("default")))

#define TZ_MAX_SQ 36
#define TZ_MAX_MOVES 1024 /* upper bound of legal moves per position handled by the library */
#define TZ_MAX_PLIES 1024 /* longest recorded replay */
#define TZ_MAX_K 64       /* largest `sampled_actions` */

/* return codes */
enum {
    TZ_OK = 0,
    TZ_EINVAL = -1,   /* bad argument (the reference would assert/panic) */
    TZ_ECUDA = -2,    /* CUDA runtime error */
    TZ_ESEARCH = -3,  /* sticky device-side search error, see tz_status() */
    TZ_ENOMEM = -4,
    TZ_ENOWEIGHTS = -5,
};

/* tz_status() bits (device-side invariant violations; the reference panics on these) */
enum {
    TZ_STATUS_ARENA_FULL = 1,      /* a game's node arena overflowed: raise arena_slots */
    TZ_STATUS_DEPTH = 2,           /* selection path longer than 256 plies */
    TZ_STATUS_NO_CHILD = 4,        /* "there should always be a child to simulate" */
    TZ_STATUS_TOO_MANY_MOVES = 8,  /* more legal moves than move_stride */
    TZ_STATUS_BAD_MOVE = 16,       /* "Action should be valid" (env.rs:44) */
    TZ_STATUS_NAN = 32,            /* NaN logit / value (net6_simhash.rs:304) */
    TZ_STATUS_SET_EMPTY = 64,      /* sequential halving on a root without children */
    TZ_STATUS_REPLAY_FULL = 128,
    TZ_STATUS_NETWORK_STALL = 256, /* a CTA pair of the fused network launch waited > ~1 s for another pair's
                                      tile (never seen; the watchdog turns a would-be hang into this error) */
    TZ_STATUS_WEIGHTS_MISMATCH = 512, /* a broadcast weight set describes another network (board size, residual
                                         blocks or 16-bit type differ between the ranks) */
    TZ_STATUS_TARGETS_FULL = 1024, /* resident self-play recording ran out of room: a game's record region (its
                                      recorded prefix is still emitted) or the output queue (whole games that do not
                                      fit are dropped); the search is not affected.  See tz_selfplay_record. */
};

/* Move (takparse `Move`, 2 bytes):
 *   bits 0..2 column (file a = 0), bits 3..5 row (rank 1 = 0),
 *   bits 6..7 placement: piece (0 flat, 1 wall, 2 cap); spread: direction (0 '+', 1 '-', 2 '<', 3 '>'),
 *   bits 8..15 spread pattern = takparse `Pattern::mask()` byte (MSB aligned); 0 for placements. */
typedef uint16_t tz_move_t;

/* Game state (fast-tak `Game<N, HALF_KOMI>` fields used by the reference: env.rs:50,62,
 * repr.rs:177-223).  N and HALF_KOMI are properties of the handle.  384 bytes. */
typedef struct tz_state_t {
    uint64_t stack[TZ_MAX_SQ]; /* bit i = colour (1 = black) of the piece at height i; square = row*N + col */
    uint8_t height[TZ_MAX_SQ];
    uint8_t top[TZ_MAX_SQ]; /* 0 flat, 1 wall, 2 cap; valid when height > 0 */
    uint8_t to_move;        /* 0 white, 1 black */
    uint8_t stones[2];
    uint8_t caps[2];
    uint8_t pad0;
    uint16_t ply;
    uint16_t reversible_plies;
    uint8_t pad1[14];
} tz_state_t;

typedef struct tz_config_t {
    int board_n;           /* 3..6 */
    int half_komi;         /* e.g. 4 for Game<6,4> */
    int n_games;           /* BATCH_SIZE of BatchedMCTS, dynamic here */
    int device;            /* CUDA ordinal */
    int game_base;         /* global id of game 0 (sharding: RNG streams are keyed by global id); 0..INT_MAX - n_games */
    int reversible_limit;  /* reversible-ply draw threshold; 0 = default 100 (unpinned, see DESIGN.md) */
    int move_stride;       /* row stride of per-game move/logit tables; 0 = default for board_n */
    uint32_t arena_slots;  /* node slots per game per arena half; 0 = sized from free HBM */
    int tree_batch;        /* search trees (tz_tree_*, tz_trees_*): leaves per network batch, all trees; 0 = n_games */
} tz_config_t;

typedef struct tz_handle tz_handle;

/* `Agent::policy_value_uncertainty` (agent.rs:5-14) as a host callback: fill un-normalised logits
 * (same order as the action lists), value and variance for `batch` positions. */
typedef void (*tz_agent_fn)(void* ctx, int batch, const tz_state_t* envs, const tz_move_t* actions,
                            const int* n_actions, int stride, float* logits, float* values,
                            float* variances);

enum {
    TZ_AGENT_SYNTHETIC = 0, /* deterministic integer-hash agent, bit-identical to the oracle's */
    TZ_AGENT_HOST = 1,      /* tz_agent_fn callback ("reference network outputs injected") */
    TZ_AGENT_NETWORK = 2,   /* the 16-bit tcgen05 ResNet on the device (tz_set_weights first) */
};

/* One named f32 tensor of the network (host memory), see tz_set_weights. */
typedef struct tz_tensor_t {
    const char* name;
    const float* data;
    const int64_t* shape;
    int ndim;
} tz_tensor_t;

typedef struct tz_counters_t {
    uint64_t simulations; /* calls of Node::forward */
    uint64_t evaluations; /* positions sent to the agent */
    uint64_t known;       /* forwards that ended in Forward::Known */
    uint64_t expansions;
} tz_counters_t;

typedef struct tz_root_t {
    uint32_t eval_tag;  /* 0 Value, 1 Win, 2 Loss, 3 Draw (eval.rs:8-13) */
    uint32_t eval_bits; /* f32 bits of the value, or the ply */
    uint32_t visit_count;
    uint32_t std_dev_bits;
    uint32_t n_children;
    uint32_t arena_used;
} tz_root_t;

/* ---- lifetime ---------------------------------------------------------------------- */
TZ_API const char* tz_last_error(void);
TZ_API const char* tz_version(void);
TZ_API int tz_create(const tz_config_t* cfg, tz_handle** out);            /* BatchedMCTS::new (batched.rs:33-47) */
TZ_API void tz_destroy(tz_handle* h);
TZ_API int tz_sync(tz_handle* h);
TZ_API int tz_status(tz_handle* h, uint32_t* out_bits);                    /* syncs; 0 bits = healthy */
TZ_API int tz_clear_status(tz_handle* h);
TZ_API int tz_info(tz_handle* h, int* out_move_stride, uint32_t* out_arena_slots, int* out_input_channels,
            int* out_output_channels);
TZ_API void* tz_host_alloc(size_t bytes);                                  /* pinned host memory */
TZ_API void tz_host_free(void* p);

/* ---- rules / encoding parity hooks (stateless) ---------------------------------------- */
/* Environment::populate_actions -> Game::possible_moves (env.rs:39-41), fast-tak order */
TZ_API int tz_legal_moves(tz_handle* h, const tz_state_t* states, int count, int stride, tz_move_t* out_moves,
                   int* out_n);
/* Environment::step -> Game::play (env.rs:43-45); out_ok[i] = 0 where the reference would panic */
TZ_API int tz_apply(tz_handle* h, tz_state_t* states, const tz_move_t* moves, int count, int* out_ok);
/* Environment::terminal (env.rs:47-59): 0 none, 1 win, 2 loss, 3 draw for the side to move */
TZ_API int tz_result(tz_handle* h, const tz_state_t* states, int count, int* out_terminal);
/* Game::result in absolute terms (the suffix of a Replay line, target.rs:226-230):
 * 0 ongoing, 1 "R-0", 2 "0-R", 3 "F-0", 4 "0-F", 5 "1/2-1/2" */
TZ_API int tz_game_result(tz_handle* h, const tz_state_t* states, int count, int* out_result);

/* ---- device draws ----------------------------------------------------------------------- */
/* Where a call takes NULL for its randomness, it draws on the device h = rng_hash(seed, a, b, c) (stated at
 * tz_training_batch) with a = game_base + g, the global game id, so sharded handles draw what one handle would:
 *   Gumbel noise (tz_gumbel_sequential_halving, tz_selfplay_move, tz_reanalyze_batch), child i of game g:
 *     b = move counter, c = i; u = ((float)(h >> 41) + 0.5f) * 2^-23, exactly (x + 1/2) * 2^-23 for the 23-bit x,
 *     in [2^-24, 1 - 2^-24]; noise = -logf(-logf(u)) in float32, finite
 *   self-play sample (tz_select_selfplay, tz_selfplay_move): b = move counter, c = 0x5e1ec; the first child whose
 *     cumulative weight exceeds h mod (total weight)
 *   opening (tz_new_openings, tz_restart_terminal, the restart of tz_selfplay_move): b = opening counter,
 *     c = 0x0fe11; sym = h & 7, adj = (h >> 3) & 1
 *   random step (tz_random_steps): b = the ply before the step, c = 0x57e95; the move h mod count of
 *     tz_legal_moves' list
 * Counters of a handle, both 0 at tz_create: the move counter goes up by one at the end of every search of
 * tz_gumbel_sequential_halving, tz_selfplay_move and tz_reanalyze_batch.  A search's noise uses the counter before it;
 * tz_select_selfplay uses the current one, so after a search the one after it; tz_selfplay_move samples with the
 * counter after its search (noise c, sample c + 1).  The opening counter goes up by one on every tz_new_openings and
 * every restart (tz_restart_terminal and inside tz_selfplay_move), whether or not a game finished. */

/* ---- positions ------------------------------------------------------------------------- */
/* BatchedMCTS::from_envs / nodes_and_envs_mut writes (reanalyze/src/main.rs:159-165); roots reset */
TZ_API int tz_set_positions(tz_handle* h, const tz_state_t* states, const uint8_t* mask);
TZ_API int tz_get_positions(tz_handle* h, tz_state_t* out);
/* Env::new_opening (env.rs:65-79); sym/adj NULL = draw from the library RNG with `seed` */
TZ_API int tz_new_openings(tz_handle* h, const uint8_t* mask, const int* sym, const int* adj, uint64_t seed);
/* the random part of Env::new_opening_with_random_steps (env.rs:81-96): `steps` uniformly random legal moves
 * in every selected game (library RNG keyed by seed / global game id / ply), roots reset */
TZ_API int tz_random_steps(tz_handle* h, const uint8_t* mask, int steps, uint64_t seed);
TZ_API int tz_reset_roots(tz_handle* h, const uint8_t* mask);              /* *node = Node::default() */

/* ---- search ----------------------------------------------------------------------------- */
TZ_API int tz_set_agent(tz_handle* h, int kind, tz_agent_fn fn, void* ctx);
/* BatchedMCTS::simulate (batched.rs:63-128) */
TZ_API int tz_simulate(tz_handle* h, const float* betas);
/* BatchedMCTS::gumbel_sequential_halving (batched.rs:207-409).  gumbel: [n_games][gumbel_stride]
 * injected Gumbel(0,1) draws, one per root child in child order, or NULL to draw them on the
 * device from `seed` (readable afterwards with tz_last_gumbel). */
TZ_API int tz_gumbel_sequential_halving(tz_handle* h, const float* betas, int sampled_actions,
                                 uint32_t search_budget, const float* gumbel, int gumbel_stride,
                                 uint64_t seed, tz_move_t* out_moves);
TZ_API int tz_last_gumbel(tz_handle* h, float* out, int stride);
/* BatchedMCTS::step (batched.rs:131-144) incl. Node::descend subtree reuse */
TZ_API int tz_step(tz_handle* h, const tz_move_t* moves);
/* BatchedMCTS::restart_terminal_envs (batched.rs:185-203); out_terminal[g] as tz_result */
TZ_API int tz_restart_terminal(tz_handle* h, const int* sym, const int* adj, uint64_t seed, int* out_terminal);
/* Replay of the game that tz_restart_terminal just finished / of the game in progress */
TZ_API int tz_finished_replay(tz_handle* h, int game, tz_state_t* out_start, tz_move_t* out_moves, int cap);
TZ_API int tz_replay(tz_handle* h, int game, tz_state_t* out_start, tz_move_t* out_moves, int cap);

/* ---- root read-backs (direct `Node` field reads of the callers) ---------------------------- */
TZ_API int tz_root_children(tz_handle* h, int stride, int* out_n, tz_move_t* moves, uint32_t* visits,
                     uint32_t* eval_tag, uint32_t* eval_bits, float* logit, float* prob, float* std_dev);
TZ_API int tz_root_stats(tz_handle* h, tz_root_t* out);
/* Node::improved_policy (policy.rs:36-48; visitations < 0 = most_visited_count()) and
 * Node::ube_target (node/mod.rs:215-230) */
TZ_API int tz_targets(tz_handle* h, float visitations, float beta, int stride, float* out_policy, float* out_ube,
               int* out_n, tz_move_t* out_moves);
/* select_best_actions / select_actions_in_selfplay (batched.rs:152-183) */
TZ_API int tz_select_best(tz_handle* h, tz_move_t* out_moves);
TZ_API int tz_select_selfplay(tz_handle* h, int weighted_random_plies, uint32_t threshold, float allowed_eval_drop,
                       const uint64_t* randoms, uint64_t seed, tz_move_t* out_moves);
TZ_API int tz_counters(tz_handle* h, tz_counters_t* out);
/* BatchedMCTS::apply_noise / Node::apply_dirichlet (batched.rs:146-151, node/noise.rs:10-26): the host mixes
 * p' = p*(1-ratio) + noise*ratio and takes logit' = ln(p') with its libm (as the reference does) from
 * tz_root_children, then stores both here: [n_games][stride], child order */
TZ_API int tz_set_root_priors(tz_handle* h, int stride, const float* prob, const float* logit);

/* One self-play move of every game without host buffers (the loop body of selfplay/src/main.rs:
 * 138-153, 238-329 minus the file I/O): search with library-drawn Gumbel noise, improved-policy /
 * UBE targets into device buffers, visit-weighted sampling on early plies, step, restart of finished
 * games.  Asynchronous: returns once enqueued; tz_sync / tz_counters / tz_status wait. */
typedef struct tz_selfplay_t {
    int sampled_actions;        /* SAMPLED_ACTIONS */
    uint32_t search_budget;     /* SEARCH_BUDGET */
    float beta;                 /* BETA for the first half of the batch (`exploration` feature), else 0 */
    int weighted_random_plies;  /* WEIGHTED_RANDOM_PLIES (10) */
    uint32_t sample_threshold;  /* 32 */
    float allowed_eval_drop;    /* 0.5 */
    float target_visitations;   /* IMPROVED_POLICY_VISITATIONS */
    float target_beta;          /* ube_target beta (0.25) */
    uint64_t seed;
} tz_selfplay_t;
TZ_API int tz_selfplay_move(tz_handle* h, const tz_selfplay_t* params);
TZ_API int tz_launch_count(tz_handle* h, uint64_t* out);             /* kernels launched so far */

/* Training data of tz_selfplay_move, kept on the device (take_a_step + restart_envs_and_complete_targets,
 * selfplay/src/main.rs:238-329).  With recording on, every tz_selfplay_move appends one pending record per game (root
 * position, replay index, improved policy in child order, UBE target) to the game's region of `bytes_per_game` bytes
 * (a record takes 400 + 6 * children bytes, rounded up to 16), and when a game ends it emits, into the output queue,
 * the game's replay and its targets from the last ply to the first with the value completed from the result
 * (exploration half, beta != 0 and game < n_games / 2: only plies > weighted_random_plies).  Finished games come in
 * ascending game order; the order does not depend on timing.
 *   bytes_per_game 0: a quarter of the free HBM divided among the games, at least 64 KiB and at most the worst case
 *     TZ_MAX_PLIES * (400 + 6 * move_stride); tz_selfplay_read reports the most any game has used.
 *   output_bytes 0: half the size of all regions, at most an eighth of the free HBM, at least 16 MiB.  The queue is
 *     split: 1/16 replays, 1/16 replay moves, the rest targets and policy entries sized for a mean of move_stride / 4
 *     children per target.
 * A full region stops that game's recording (its prefix is still emitted with correct values); whole games that do
 * not fit the queue are dropped; both raise TZ_STATUS_TARGETS_FULL and never disturb the search.  Pending records
 * belong to consecutive tz_selfplay_move calls: tz_step, tz_restart_terminal, tz_new_openings, tz_set_positions,
 * tz_random_steps, tz_reset_roots, tz_reanalyze_batch with indices and the tz_tree_* calls drop them at the next
 * recording move.  enable = 0 frees everything; enabling again starts empty.  Recording off (the default) leaves
 * tz_selfplay_move's launches exactly as they are. */
TZ_API int tz_selfplay_record(tz_handle* h, int enable, size_t bytes_per_game, size_t output_bytes);

/* Caller buffers of tz_selfplay_read.  The caller sets the four capacities (entries) and any of the pointers (NULL
 * skips that field); the call sets the counts. */
typedef struct tz_selfplay_data_t {
    size_t target_cap;
    size_t policy_cap;
    size_t replay_cap;
    size_t move_cap;
    tz_state_t* target_env;       /* [targets] position before the move */
    float* target_value;          /* [targets] value target */
    float* target_ube;            /* [targets] UBE target */
    int* target_n;                /* [targets] policy entries */
    uint64_t* target_offset;      /* [targets] first entry in policy_moves / policy_probs */
    int* target_game;             /* [targets] global game id (game_base + game) */
    tz_move_t* policy_moves;      /* [policy] */
    float* policy_probs;          /* [policy] improved policy */
    tz_state_t* replay_start;     /* [replays] start position */
    int* replay_result;           /* [replays] tz_game_result code of the final position */
    int* replay_terminal;         /* [replays] tz_result code of the final position */
    int* replay_length;           /* [replays] moves */
    uint64_t* replay_offset;      /* [replays] first move in replay_moves */
    int* replay_game;             /* [replays] global game id */
    uint8_t* replay_exploration;  /* [replays] 1 for the exploration half */
    tz_move_t* replay_moves;      /* [moves] */
    size_t n_targets;             /* out: entries returned, or needed when a capacity is too small */
    size_t n_policy;
    size_t n_replays;
    size_t n_moves;
    size_t high_water_bytes;      /* out: most bytes one game's region has held since tz_selfplay_record */
} tz_selfplay_data_t;
/* Waits for the handle's stream, copies the queue out (cudaMemcpyAsync on the handle's stream) and empties it.  A
 * capacity below its count returns TZ_EINVAL with the counts set and consumes nothing; TZ_ESEARCH on a device search
 * error (TZ_STATUS_TARGETS_FULL is not one). */
TZ_API int tz_selfplay_read(tz_handle* h, tz_selfplay_data_t* io);

/* ---- training batches on the device (the data side of `learn`: replay buffer, Augment, game_to_tensor,
 * policy_tensor / move_mask, target.rs:32-54, repr.rs:169-244) ------------------------------------------------------
 *
 * Target buffer: a FIFO ring of `capacity` targets in device memory.  Every slot has a fixed stride: the position
 * (384 B), value, UBE target and entry count (12 B) and move_stride (move, probability) pairs (6 B each), so a slot
 * takes 396 + 6 * move_stride bytes: about 6.5 KB for the 6x6 default stride of 1024, 6.5 GB for 10^6 targets.  A
 * root never has more than move_stride children, so a slot cannot overflow.  TZ_ENOMEM when it does not fit; capacity
 * 0 frees the buffer; calling again replaces it with an empty one.  When the ring is full the oldest targets are
 * overwritten.
 *   from_selfplay = 1: while recording is on (tz_selfplay_record), every target tz_selfplay_move emits into the output
 *     queue is also appended, device to device and in queue order (finished games ascending, each from its last ply to
 *     its first; the exploration filter applies; games dropped under TZ_STATUS_TARGETS_FULL are in neither).  The
 *     queue, tz_selfplay_read and the search are unchanged.  With from_selfplay = 0 or no buffer, tz_selfplay_move
 *     launches exactly what it launches without one. */
TZ_API int tz_target_buffer(tz_handle* h, size_t capacity, int from_selfplay);
/* Appends `count` targets from host arrays in the layout tz_selfplay_read returns: target i is env[i], value[i],
 * ube[i] and the n[i] entries moves / probs[offset[i] .. offset[i] + n[i]) of arrays holding n_policy entries.
 * TZ_EINVAL, appending nothing, when n[i] < 0 or n[i] > move_stride, an entry range falls outside n_policy, a move
 * has no move_index on this board size (square off the board, placement of a piece code above 2, spread pattern that
 * does not fit N), a target lists the same move twice (both would land on one policy index), or a position is not one
 * of this board.  Waits for the handle's stream. */
TZ_API int tz_target_buffer_append(tz_handle* h, size_t count, const tz_state_t* env, const float* value,
                                   const float* ube, const int* n, const uint64_t* offset, const tz_move_t* moves,
                                   const float* probs, size_t n_policy);
/* Waits for the handle's stream; *size = targets kept (at most the capacity), *appended = targets ever appended since
 * tz_target_buffer (for replay-ratio accounting).  Either pointer may be NULL. */
TZ_API int tz_target_buffer_info(tz_handle* h, size_t* size, uint64_t* appended);

/* One training batch: `batch` examples from the target buffer, written into CALLER-OWNED DEVICE MEMORY (every
 * non-NULL output must be device memory of the handle's device).  C = 2 * (2N + 5) + 2 input channels and
 * OC = 3 + 4 * (2^N - 2) output channels, as tz_info reports them.
 * Example i takes target index[i] (counted from the oldest kept target) under symmetry sym[i]:
 *   index[i] = indices ? indices[i] : high 64 bits of (rng_hash(seed, i, 0, 0) * size)
 *   sym[i]   = symmetry ? symmetry[i] : augment ? rng_hash(seed, i, 1, 0) & 7 : 0
 * with rng_hash(s, a, b, c) = mix(mix(mix(mix(s ^ 0x9e3779b97f4a7c15) ^ a * 0xbf58476d1ce4e5b9) ^ b *
 * 0x94d049bb133111eb) ^ c * 0xd6e8feb86659fd93) and mix the murmur3 64-bit finalizer (x ^= x >> 33;
 * x *= 0xff51afd7ed558ccd; x ^= x >> 33; x *= 0xc4ceb9fe1a85ec53; x ^= x >> 33), all modulo 2^64.
 * A symmetry maps square (row, col) by, in this order: bit 0 mirrors the column, bit 1 mirrors the row, bit 2 swaps
 * row and column (the order of tz_new_openings).  A spread keeps its pattern byte; its direction is mapped in the same
 * order: bit 0 swaps '<' and '>', bit 1 swaps '+' and '-', bit 2 swaps '+' with '>' and '-' with '<'.  Reserves, side
 * to move, ply and reversible plies are kept.
 *   planes   f32 [batch][C][N][N]  game_repr of the transformed position (the encoding of tz_encode_planes)
 *   policy   f32 [batch][OC][N][N] zero, and each entry's probability at move_index of the transformed move
 *   mask     u8  [batch][OC][N][N] 1 at the same places, 0 elsewhere
 *   value, ube    f32 [batch]       the target's, unchanged
 *   out_index, out_symmetry i32 [batch]  what was used
 * Waits for the handle's stream (queued self-play appends land first), then validates: TZ_EINVAL for an empty
 * buffer, batch <= 0, an index at or past the size, a symmetry above 7 or an output that is not device memory of the
 * handle's device.  Asynchronous: returns once the kernel is enqueued on the handle's stream; tz_sync waits. */
typedef struct tz_training_batch_t {
    int batch;
    const uint64_t* indices;  /* host [batch] or NULL: drawn */
    const int* symmetry;      /* host [batch] 0..7 or NULL: drawn when augment, else 0 */
    int augment;
    uint64_t seed;
    float* planes;            /* device outputs; NULL skips */
    float* policy;
    uint8_t* mask;
    float* value;
    float* ube;
    int* out_index;           /* i32 */
    int* out_symmetry;
} tz_training_batch_t;
TZ_API int tz_training_batch(tz_handle* h, const tz_training_batch_t* params);
/* `update_counts` (net6_simhash.rs:236-241) for a batch that stays on the device: reads only batch, indices, symmetry,
 * augment and seed of `params` (the outputs are ignored), resolves example i's target index and symmetry exactly as
 * tz_training_batch does (explicit arrays or the rng_hash draws above), and marks, in the handle's novelty set, the
 * hash index (the hash set last: SimHash or LCG) of that target's position under that symmetry.  A learner passes the
 * params of the batch it just trained on.  Which form the reference's `learn` marks -- the augmented position it
 * trained on or the position as stored -- was not checked against the reference: the caller chooses, through
 * symmetry / augment; augment = 0 (or all-zero symmetries) marks the positions as stored.
 * Validation and codes as tz_training_batch (waits for the stream, then TZ_EINVAL for an empty buffer, batch <= 0, an
 * index at or past the size or a symmetry above 7, nothing marked); TZ_ENOWEIGHTS without tz_set_simhash /
 * tz_set_lcghash.  A set that is still the empty one of a fresh network becomes a real, zeroed one first (as in
 * tz_update_counts).  Asynchronous: one kernel on the handle's stream, so on a self-play handle the marks land between
 * the moves enqueued before and after the call. */
TZ_API int tz_update_counts_buffer(tz_handle* h, const tz_training_batch_t* params);

/* The loop body of `reanalyze` (reanalyze/src/main.rs:147-235) without per-batch host buffers.  tz_stage_positions
 * uploads the positions of the replay buffer once (position_buffer, main.rs:60-75); tz_reanalyze_batch makes the
 * staged positions pool_indices[g] the fresh roots of the games (`*node = Node::default(); *env = replay_env`, NULL =
 * keep the current positions / roots, e.g. after tz_set_positions), searches them (ZERO_BETA, library-drawn Gumbel
 * noise) and leaves the targets on the device: improved policy at most_visited_count() visitations, UBE target, and
 * the value target (root evaluation when known, else the negated evaluation of the selected child, main.rs:184-195).
 * Asynchronous like tz_selfplay_move; tz_reanalyze_read copies the targets of the last batch out. */
typedef struct tz_reanalyze_t {
    int sampled_actions;    /* SAMPLED_ACTIONS */
    uint32_t search_budget; /* SEARCH_BUDGET */
    float target_beta;      /* UBE_TARGET_BETA */
    uint64_t seed;
} tz_reanalyze_t;
TZ_API int tz_stage_positions(tz_handle* h, const tz_state_t* states, size_t count);
TZ_API int tz_reanalyze_batch(tz_handle* h, const uint32_t* pool_indices, const tz_reanalyze_t* params);
TZ_API int tz_reanalyze_read(tz_handle* h, int stride, float* out_policy, float* out_ube, float* out_value, int* out_n,
                      tz_move_t* out_moves);

/* Sampled per-kernel device timing: every `sample_every`-th lock-step simulation is bracketed with
 * CUDA events on the library's stream.  Categories: 0 select(+movegen,+known backup), 1 encode,
 * 2 input conv, 3 tower convs, 4 policy conv, 5 heads+gather, 6 expand(+softmax,+backup), 7 synthetic agent. */
typedef struct tz_profile_t {
    double ms[8];
    uint64_t launches[8];
    uint64_t locksteps; /* sampled lock-step simulations */
    uint64_t positions; /* positions evaluated in the sampled lock-steps */
} tz_profile_t;
TZ_API int tz_profile_begin(tz_handle* h, int sample_every);
TZ_API int tz_profile_end(tz_handle* h, tz_profile_t* out);
/* CUDA-event stopwatch on the library's stream: start is asynchronous, stop waits and returns ms */
TZ_API int tz_timer_start(tz_handle* h);
TZ_API int tz_timer_stop(tz_handle* h, double* out_ms);

/* ---- single tree (tei/src/main.rs:139-290, analysis/src/main.rs): the tree and position are game 0 of the
 * handle (tz_set_positions / tz_reset_roots); batch_size <= max(n_games, tree_batch). -------------------------- */
TZ_API int tz_tree_simulate_simple(tz_handle* h, float beta);                 /* Node::simulate_simple (mcts.rs:235-266) */
TZ_API int tz_tree_simulate_batch(tz_handle* h, float beta, int batch_size);  /* Node::simulate_batch (mcts.rs:268-328) */
TZ_API int tz_tree_descend(tz_handle* h, tz_move_t move);                     /* Node::descend + env.step (tree reuse) */
/* Node::principal_variation (node/mod.rs:40-62); returns the length written to out_moves */
TZ_API int tz_tree_principal_variation(tz_handle* h, tz_move_t* out_moves, int cap);

/* ---- many single trees at once: the tree of every selected game (mask [n_games], NULL = every game), each with the
 * single-tree semantics above, searched side by side.  A mask that selects no game is a no-op.  Like tz_tree_*,
 * these calls make pending self-play records stale. ---------------------------------------------------------------- */
/* Node::simulate_batch (mcts.rs:268-328) on every selected game's tree at once: each tree gets up to batch_size leaves
 * (4 * batch_size forwards), one network batch for all of them.  Selected games * batch_size <= max(n_games, tree_batch). */
TZ_API int tz_trees_simulate_batch(tz_handle* h, const uint8_t* mask, float beta, int batch_size);
/* Node::descend + env.step per selected game (moves [n_games]; entries of unselected games are ignored) */
TZ_API int tz_trees_descend(tz_handle* h, const uint8_t* mask, const tz_move_t* moves);
/* Node::principal_variation per game: out_moves [n_games][cap], out_len [n_games] (0 for unselected games); entries of
 * out_moves past a game's length are left as they were */
TZ_API int tz_trees_principal_variation(tz_handle* h, const uint8_t* mask, int cap, tz_move_t* out_moves, int* out_len);

/* ---- network (takzero/src/network/{net4_simhash,net5,net6_simhash,residual,repr}.rs) ----------- */
/* Net::load (network/mod.rs:16-35): f32 tensors in PyTorch layout, named
 *   core.input_conv2d.weight [256,C,3,3]; core.batch_norm.{weight,bias,running_mean,running_var} [256];
 *   core.res_block_{b}.{0,1}.conv2d.weight [256,256,3,3]; core.res_block_{b}.{0,1}.batch_norm.* [256];
 *   policy.conv2d.{weight [O,256,3,3], bias [O]}; {value,ube}.conv2d.{weight [1,256,1,1], bias [1]};
 *   {value,ube}.linear.{weight [1,N*N], bias [1]}.
 * The number of residual blocks is taken from the names (16 for net4/net6, 20 for net5).  BatchNorm is
 * folded (eval mode, eps 1e-5) and the convolutions are converted to the 16-bit network type here.
 * A 5x5 model's RND estimator (net5.rs:120-146,193-211) rides along when its tensors are present:
 *   {rnd_learning,rnd_target}.{input_linear [1024,C*N*N], hidden_linear [1024,1024], final_linear [512,1024]}.{weight,bias},
 *   min [1], max [1]; the local uncertainty is then normalized_rnd instead of the hash-set lookup. */
TZ_API int tz_set_weights(tz_handle* h, const tz_tensor_t* tensors, int count);

/* ---- multi-GPU (one process per GPU; games shard by contiguous global id, tz_config_t::game_base) ------------
 * The reference scales by independent `selfplay` processes that share files (README.md:128-130): each re-reads
 * `model_latest.ot` before every move (selfplay/src/main.rs:107) and `learn` adds up what they produced through
 * `buffer_lengths.txt` (learn/src/main.rs:195-209).  Here those two exchanges are NCCL collectives over NVLink; there
 * is none inside a simulation.  NCCL is opened at run time (TZ_NCCL_LIB or libnccl.so.2); a single-GPU host needs none.
 *
 * tz_comm_unique_id: 128 bytes (an ncclUniqueId) made by one rank and handed to the others by the host's own means;
 * tz_comm_init: collective over all `nranks` ranks (nranks == 1: no NCCL involved). */
TZ_API int tz_comm_unique_id(void* out_id128);
TZ_API int tz_comm_init(tz_handle* h, const void* id128, int nranks, int rank);
TZ_API int tz_comm_destroy(tz_handle* h);
/* One weight GENERATION on every rank of the communicator (collective; also valid without one = Net::load on a single
 * GPU): the root rank passes the model's tensors (as tz_set_weights), folds BatchNorm and arranges the 16-bit weight
 * image on its GPU, ncclBroadcast sends that image (39 MB for the 6x6 network) into the inactive one of every rank's two
 * weight sets, and every rank swaps sets for the launches it enqueues from then on -- i.e. between two moves.  All of
 * it runs on a side stream beside the search.  The other ranks pass tensors = NULL and the number of residual blocks
 * (0 = the board's default: 20 for 5x5, else 16); every rank must use the same tz_set_network_dtype.  Tensor data in
 * pinned memory (tz_host_alloc) is uploaded from where it is, asynchronously: leave it unchanged until
 * tz_weight_generation has returned; data in pageable memory is copied into the library's own staging buffer before
 * the call returns (the same holds for tz_set_weights).  The RND estimator of a 5x5 model is not part of the image: the
 * root takes it from its tensors as tz_set_weights does (a model without it switches it off), the other ranks keep
 * the one they had. */
TZ_API int tz_broadcast_weights(tz_handle* h, const tz_tensor_t* tensors, int count, int res_blocks, int root);
/* One novelty-set GENERATION on every rank of the communicator (collective; without one, or with nranks == 1, a set
 * generation on one GPU): the 512 MiB set travels like the weight image of tz_broadcast_weights -- written into the
 * inactive one of two sets on the same side stream, ncclBroadcast to the inactive set of every other rank, swapped for
 * the launches each rank enqueues afterwards; launches already enqueued keep reading the old set.  The second set is
 * allocated by the first call (a handle that never calls this holds one set).  Every rank needs a network
 * (TZ_ENOWEIGHTS otherwise).  The root's `bitset`:
 *   a host image in the bitvec.bin layout (2^29 bytes, LSB-first) in pinned memory (tz_host_alloc): uploaded from
 *     where it is, asynchronously; leave it unchanged until tz_sync
 *   a host image in pageable memory: copied before the call returns, through a 16 MiB pinned staging buffer of the
 *     handle (the call then waits until the readers of the set it overwrites, the launches enqueued before the last
 *     swap, have run)
 *   NULL: the root's own current set, marks of tz_update_counts / tz_update_counts_buffer enqueued before the call
 *     included (the copy waits for them on the device)
 * The other ranks pass NULL.  The root needs a hash (tz_set_simhash / tz_set_lcghash, else TZ_ENOWEIGHTS); the
 * broadcast carries its hash kind and board size, and a rank whose hash differs, or that has none, raises
 * TZ_STATUS_WEIGHTS_MISMATCH on the device and keeps its old set.  The SimHash matrix / LCG multipliers are not
 * broadcast: they come with the model (tz_set_simhash, tz_set_lcghash, tz_load_model), as before.  TZ_EINVAL, nothing
 * changed, for a root out of range or a non-NULL bitset on another rank.  Sets are not OR-reduced over ranks: the
 * root's set is the set (one learner). */
TZ_API int tz_broadcast_novelty_set(tz_handle* h, const uint8_t* bitset, int root);
/* number of generations so far and the device time of the last one (upload + fold + broadcast); waits for it */
TZ_API int tz_weight_generation(tz_handle* h, uint64_t* out_generation, double* out_ms);
/* in-place sum over all ranks of up to 64 counters (simulations, positions, targets, finished games ...) */
TZ_API int tz_allreduce_sum(tz_handle* h, uint64_t* values, int count);
/* Net::load (network/mod.rs:20-27, net6_simhash.rs:164-181) from the reference's own model file: `path` is a tch
 * `VarStore::save` archive (`model_latest.ot`, written by learn/src/main.rs:166,257 and re-read before every move
 * by selfplay/src/main.rs:107 and reanalyze/src/main.rs:93), parsed here without libtorch (ZIP + pickle); a
 * `torch.save` state dict, a safetensors file (what tch writes for a ".safetensors" path) or this repository's
 * TZW1 container work too.  tch variable names are mapped to the
 * names above: the two SmallBlocks of a ResidualBlock share one path (residual.rs:52-54), so the file holds
 * `core.res_block_B.conv2d.weight` (block half 0) and `core.res_block_B.conv2d.weight__K` (half 1).  When the file
 * has a `simhash_matrix` (or `lcghash_init`), it and the sidecar `bitvec.bin` next to the file go through
 * tz_set_simhash (tz_set_lcghash).  Like Net::load, tz_load_model fails when the sidecar is missing;
 * tz_load_model_ex(allow_missing_set = 1) takes a missing sidecar as the empty set of a freshly initialised network
 * (every local uncertainty is then MAXIMUM_VARIANCE = 4.0). */
TZ_API int tz_load_model(tz_handle* h, const char* path);
TZ_API int tz_load_model_ex(tz_handle* h, const char* path, int allow_missing_set);
/* Tensor::load_multi: calls fn for every tensor of the file (converted to contiguous f32) with the mapped and the
 * stored name; returns the tensor count or a negative code.  Needs no GPU. */
typedef void (*tz_model_tensor_fn)(void* ctx, const char* name, const char* stored_name, const float* data,
                                   const int64_t* shape, int ndim);
TZ_API int tz_read_model_file(const char* path, tz_model_tensor_fn fn, void* ctx);
/* 16-bit type the NEXT tz_set_weights / tz_load_model converts weights and activations to; both run the same tcgen05
 * kind::f16 kernels.  TZ_DTYPE_F16 (IEEE half, the default) is the mode whose whole searches choose the same move as
 * the f32 reference network on >= 99 % of positions (tests/test_gpu_agreement.py); range 65504: an overflow surfaces
 * as TZ_STATUS_NAN.  TZ_DTYPE_BF16 has 3 fewer mantissa bits (~8x the error, ~97.5 % agreement) and is a few per
 * cent faster under the power cap. */
enum { TZ_DTYPE_BF16 = 0, TZ_DTYPE_F16 = 1 };
TZ_API int tz_set_network_dtype(tz_handle* h, int dtype);
/* `impl Agent for Net`::policy_value_uncertainty (net6_simhash.rs:259-324) on host buffers:
 * count <= n_games positions, actions [count][stride] -> logits [count][stride], values, variances */
TZ_API int tz_evaluate(tz_handle* h, const tz_state_t* states, int count, const tz_move_t* actions,
                const int* n_actions, int stride, float* logits, float* values, float* variances);
/* SimHash novelty (net6_simhash.rs:136-139,203-256): matrix [C*N*N][32] f32 and the optional 2^32-bit set
 * (the 512 MiB `bitvec.bin` sidecar of the model, LSB-first); bitset NULL = empty set (fresh network), for
 * which the local uncertainty is MAXIMUM_VARIANCE = 4.0.  tz_simhash_indices = `get_indices` (parity hook). */
TZ_API int tz_set_simhash(tz_handle* h, const float* matrix, const uint8_t* bitset);
TZ_API int tz_simhash_indices(tz_handle* h, const tz_state_t* states, int count, uint32_t* out);
/* LCG-hash novelty (net4_lcghash.rs:131-137,203-241): `lcghash_init` [C][N][N] f32 and the optional set; replaces
 * the SimHash lookup of the handle.  tz_lcghash_indices = `get_indices` (integer hash: bit-exact parity hook). */
TZ_API int tz_set_lcghash(tz_handle* h, const float* init, const uint8_t* bitset);
TZ_API int tz_lcghash_indices(tz_handle* h, const tz_state_t* states, int count, uint32_t* out);
/* `update_counts` (net6_simhash.rs:236-241; net4_lcghash.rs has the same): the hash index of every given position is
 * marked as seen in the handle's set, with the hash set last (SimHash or LCG).  A handle whose set is still the empty
 * one of a fresh network gets a real, zeroed set first.  tz_read_novelty_set copies the 2^29-byte image out in the
 * layout of the reference's `bitvec.bin` (what `Net::save` writes next to the model, net6_simhash.rs:152-170). */
TZ_API int tz_update_counts(tz_handle* h, const tz_state_t* states, int count);
TZ_API int tz_read_novelty_set(tz_handle* h, uint8_t* out, size_t cap);
/* game_repr (repr.rs:169-228): f32 planes [count][C][N][N] */
TZ_API int tz_encode_planes(tz_handle* h, const tz_state_t* states, int count, float* out);
/* test hooks: stop the tower after `limit` convolutions (-1 = full network); read back an activation
 * buffer (0 block stream, 1 block middle: f32 [count][N*N][256]) of the last tz_evaluate, or (2) the 16-bit input
 * planes the first convolution encodes from those positions, f32 [count][N*N][64] */
TZ_API int tz_debug_layer_limit(tz_handle* h, int limit);
TZ_API int tz_debug_activations(tz_handle* h, int which, int count, float* out);
/* test hook, needs no GPU: the work-item schedule of the fused network launch (conv_tcgen05.cuh `Schedule`) for
 * `count` positions -- out[0..3] = items, chunks, pair tiles per chunk, rows per chunk -- next to the bounds the
 * host sizes buffers with for `count_max` positions -- out[4..6] = chunks, pair tiles per chunk, rows of one
 * activation set; out_items receives (chunk, layer, pair tile) of the first `cap` items */
TZ_API int tz_debug_schedule(int count, int count_max, int board_n, int chunk_min_tiles, int layers, long long* out,
                      int* out_items, int cap);
/* test / measurement hook, read by the NEXT tz_set_weights (launch structure) or at once (drop_progress):
 * per_layer_launches = 1: one launch per convolution instead of the fused launch; chunk_min_tiles: minimum pair tiles
 * per chunk (-1 = default 150, 0 = one chunk); drop_progress = 1: CTA pair 0 withholds its tiles so that the watchdog
 * (TZ_STATUS_NETWORK_STALL) can be tested.  The defaults (0, -1, 0) are the product. */
TZ_API int tz_debug_network_mode(tz_handle* h, int per_layer_launches, int chunk_min_tiles, int drop_progress);
/* Test hook of the single-tree path: the descents and the backups of a batch run as in-order wavefronts of up to 8
 * warps (kernels.cu, k_tree_forward / k_tree_backward); fewer warps change the interleaving, never the result.
 * 0 = default (8). */
TZ_API int tz_debug_tree_warps(tz_handle* h, int warps);
/* parity hook: the active weight set (folded, arranged 16-bit weights + biases; layout in nn.cu `SetLayout`);
 * out = NULL: only the size */
TZ_API int tz_debug_weight_set(tz_handle* h, uint8_t* out, size_t cap, size_t* out_size);
/* parity hook: the exp of the device's softmax (policy.rs:10-19; glibc's expf algorithm restated, see DESIGN.md) */
TZ_API int tz_debug_expf(tz_handle* h, const float* in, int count, float* out);
/* tuning hook: mean ms per tower-convolution launch over `count` positions (CUDA events, `reps` blocks) */
TZ_API int tz_debug_time_tower(tz_handle* h, int count, int reps, double* ms_per_conv);

#ifdef __cplusplus
}
#endif
#endif
