//! Raw bindings of libtakzero_b200.so, GENERATED from include/takzero_b200.h by tools/gen_rust_bindings.py.
//! UNVERIFIED: the image this was produced in has no Rust toolchain; the file is checked against the header
//! (every exported tz_* function, struct and constant is present with the mapped types) but was never compiled.
//! Link with `cargo:rustc-link-lib=dylib=takzero_b200` (see INTEGRATION.md).
#![allow(non_camel_case_types, non_upper_case_globals, dead_code)]
use core::ffi::{c_char, c_int, c_longlong, c_void};

pub type tz_move_t = u16;
#[repr(C)] pub struct tz_handle { _private: [u8; 0] }

pub const TZ_MAX_SQ: usize = 36;
pub const TZ_MAX_MOVES: usize = 1024;
pub const TZ_MAX_PLIES: usize = 1024;
pub const TZ_MAX_K: usize = 64;
pub const TZ_OK: c_int = 0;
pub const TZ_EINVAL: c_int = -1;
pub const TZ_ECUDA: c_int = -2;
pub const TZ_ESEARCH: c_int = -3;
pub const TZ_ENOMEM: c_int = -4;
pub const TZ_ENOWEIGHTS: c_int = -5;
pub const TZ_STATUS_ARENA_FULL: u32 = 1;
pub const TZ_STATUS_DEPTH: u32 = 2;
pub const TZ_STATUS_NO_CHILD: u32 = 4;
pub const TZ_STATUS_TOO_MANY_MOVES: u32 = 8;
pub const TZ_STATUS_BAD_MOVE: u32 = 16;
pub const TZ_STATUS_NAN: u32 = 32;
pub const TZ_STATUS_SET_EMPTY: u32 = 64;
pub const TZ_STATUS_REPLAY_FULL: u32 = 128;
pub const TZ_STATUS_NETWORK_STALL: u32 = 256;
pub const TZ_STATUS_WEIGHTS_MISMATCH: u32 = 512;
pub const TZ_STATUS_TARGETS_FULL: u32 = 1024;
pub const TZ_AGENT_SYNTHETIC: u32 = 0;
pub const TZ_AGENT_HOST: u32 = 1;
pub const TZ_AGENT_NETWORK: u32 = 2;
pub const TZ_DTYPE_BF16: u32 = 0;
pub const TZ_DTYPE_F16: u32 = 1;

#[repr(C)]
#[derive(Clone, Copy)]
pub struct tz_state_t {
    pub stack: [u64; TZ_MAX_SQ],
    pub height: [u8; TZ_MAX_SQ],
    pub top: [u8; TZ_MAX_SQ],
    pub to_move: u8,
    pub stones: [u8; 2],
    pub caps: [u8; 2],
    pub pad0: u8,
    pub ply: u16,
    pub reversible_plies: u16,
    pub pad1: [u8; 14],
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct tz_config_t {
    pub board_n: c_int,
    pub half_komi: c_int,
    pub n_games: c_int,
    pub device: c_int,
    pub game_base: c_int,
    pub reversible_limit: c_int,
    pub move_stride: c_int,
    pub arena_slots: u32,
    pub tree_batch: c_int,
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct tz_tensor_t {
    pub name: *const c_char,
    pub data: *const f32,
    pub shape: *const i64,
    pub ndim: c_int,
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct tz_counters_t {
    pub simulations: u64,
    pub evaluations: u64,
    pub known: u64,
    pub expansions: u64,
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct tz_root_t {
    pub eval_tag: u32,
    pub eval_bits: u32,
    pub visit_count: u32,
    pub std_dev_bits: u32,
    pub n_children: u32,
    pub arena_used: u32,
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct tz_selfplay_t {
    pub sampled_actions: c_int,
    pub search_budget: u32,
    pub beta: f32,
    pub weighted_random_plies: c_int,
    pub sample_threshold: u32,
    pub allowed_eval_drop: f32,
    pub target_visitations: f32,
    pub target_beta: f32,
    pub seed: u64,
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct tz_selfplay_data_t {
    pub target_cap: usize,
    pub policy_cap: usize,
    pub replay_cap: usize,
    pub move_cap: usize,
    pub target_env: *mut tz_state_t,
    pub target_value: *mut f32,
    pub target_ube: *mut f32,
    pub target_n: *mut c_int,
    pub target_offset: *mut u64,
    pub target_game: *mut c_int,
    pub policy_moves: *mut tz_move_t,
    pub policy_probs: *mut f32,
    pub replay_start: *mut tz_state_t,
    pub replay_result: *mut c_int,
    pub replay_terminal: *mut c_int,
    pub replay_length: *mut c_int,
    pub replay_offset: *mut u64,
    pub replay_game: *mut c_int,
    pub replay_exploration: *mut u8,
    pub replay_moves: *mut tz_move_t,
    pub n_targets: usize,
    pub n_policy: usize,
    pub n_replays: usize,
    pub n_moves: usize,
    pub high_water_bytes: usize,
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct tz_reanalyze_t {
    pub sampled_actions: c_int,
    pub search_budget: u32,
    pub target_beta: f32,
    pub seed: u64,
}
#[repr(C)]
#[derive(Clone, Copy)]
pub struct tz_profile_t {
    pub ms: [f64; 8],
    pub launches: [u64; 8],
    pub locksteps: u64,
    pub positions: u64,
}

pub type tz_agent_fn = Option<unsafe extern "C" fn(ctx: *mut c_void, batch: c_int, envs: *const tz_state_t, actions: *const tz_move_t, n_actions: *const c_int, stride: c_int, logits: *mut f32, values: *mut f32, variances: *mut f32)>;
pub type tz_model_tensor_fn = Option<unsafe extern "C" fn(ctx: *mut c_void, name: *const c_char, stored_name: *const c_char, data: *const f32, shape: *const i64, ndim: c_int)>;

extern "C" {
    pub fn tz_last_error() -> *const c_char;
    pub fn tz_version() -> *const c_char;
    pub fn tz_create(cfg: *const tz_config_t, out: *mut *mut tz_handle) -> c_int;
    pub fn tz_destroy(h: *mut tz_handle);
    pub fn tz_sync(h: *mut tz_handle) -> c_int;
    pub fn tz_status(h: *mut tz_handle, out_bits: *mut u32) -> c_int;
    pub fn tz_clear_status(h: *mut tz_handle) -> c_int;
    pub fn tz_info(h: *mut tz_handle, out_move_stride: *mut c_int, out_arena_slots: *mut u32, out_input_channels: *mut c_int, out_output_channels: *mut c_int) -> c_int;
    pub fn tz_host_alloc(bytes: usize) -> *mut c_void;
    pub fn tz_host_free(p: *mut c_void);
    pub fn tz_legal_moves(h: *mut tz_handle, states: *const tz_state_t, count: c_int, stride: c_int, out_moves: *mut tz_move_t, out_n: *mut c_int) -> c_int;
    pub fn tz_apply(h: *mut tz_handle, states: *mut tz_state_t, moves: *const tz_move_t, count: c_int, out_ok: *mut c_int) -> c_int;
    pub fn tz_result(h: *mut tz_handle, states: *const tz_state_t, count: c_int, out_terminal: *mut c_int) -> c_int;
    pub fn tz_game_result(h: *mut tz_handle, states: *const tz_state_t, count: c_int, out_result: *mut c_int) -> c_int;
    pub fn tz_set_positions(h: *mut tz_handle, states: *const tz_state_t, mask: *const u8) -> c_int;
    pub fn tz_get_positions(h: *mut tz_handle, out: *mut tz_state_t) -> c_int;
    pub fn tz_new_openings(h: *mut tz_handle, mask: *const u8, sym: *const c_int, adj: *const c_int, seed: u64) -> c_int;
    pub fn tz_random_steps(h: *mut tz_handle, mask: *const u8, steps: c_int, seed: u64) -> c_int;
    pub fn tz_reset_roots(h: *mut tz_handle, mask: *const u8) -> c_int;
    pub fn tz_set_agent(h: *mut tz_handle, kind: c_int, fn_: tz_agent_fn, ctx: *mut c_void) -> c_int;
    pub fn tz_simulate(h: *mut tz_handle, betas: *const f32) -> c_int;
    pub fn tz_gumbel_sequential_halving(h: *mut tz_handle, betas: *const f32, sampled_actions: c_int, search_budget: u32, gumbel: *const f32, gumbel_stride: c_int, seed: u64, out_moves: *mut tz_move_t) -> c_int;
    pub fn tz_last_gumbel(h: *mut tz_handle, out: *mut f32, stride: c_int) -> c_int;
    pub fn tz_step(h: *mut tz_handle, moves: *const tz_move_t) -> c_int;
    pub fn tz_restart_terminal(h: *mut tz_handle, sym: *const c_int, adj: *const c_int, seed: u64, out_terminal: *mut c_int) -> c_int;
    pub fn tz_finished_replay(h: *mut tz_handle, game: c_int, out_start: *mut tz_state_t, out_moves: *mut tz_move_t, cap: c_int) -> c_int;
    pub fn tz_replay(h: *mut tz_handle, game: c_int, out_start: *mut tz_state_t, out_moves: *mut tz_move_t, cap: c_int) -> c_int;
    pub fn tz_root_children(h: *mut tz_handle, stride: c_int, out_n: *mut c_int, moves: *mut tz_move_t, visits: *mut u32, eval_tag: *mut u32, eval_bits: *mut u32, logit: *mut f32, prob: *mut f32, std_dev: *mut f32) -> c_int;
    pub fn tz_root_stats(h: *mut tz_handle, out: *mut tz_root_t) -> c_int;
    pub fn tz_targets(h: *mut tz_handle, visitations: f32, beta: f32, stride: c_int, out_policy: *mut f32, out_ube: *mut f32, out_n: *mut c_int, out_moves: *mut tz_move_t) -> c_int;
    pub fn tz_select_best(h: *mut tz_handle, out_moves: *mut tz_move_t) -> c_int;
    pub fn tz_select_selfplay(h: *mut tz_handle, weighted_random_plies: c_int, threshold: u32, allowed_eval_drop: f32, randoms: *const u64, seed: u64, out_moves: *mut tz_move_t) -> c_int;
    pub fn tz_counters(h: *mut tz_handle, out: *mut tz_counters_t) -> c_int;
    pub fn tz_set_root_priors(h: *mut tz_handle, stride: c_int, prob: *const f32, logit: *const f32) -> c_int;
    pub fn tz_selfplay_move(h: *mut tz_handle, params: *const tz_selfplay_t) -> c_int;
    pub fn tz_launch_count(h: *mut tz_handle, out: *mut u64) -> c_int;
    pub fn tz_selfplay_record(h: *mut tz_handle, enable: c_int, bytes_per_game: usize, output_bytes: usize) -> c_int;
    pub fn tz_selfplay_read(h: *mut tz_handle, io: *mut tz_selfplay_data_t) -> c_int;
    pub fn tz_stage_positions(h: *mut tz_handle, states: *const tz_state_t, count: usize) -> c_int;
    pub fn tz_reanalyze_batch(h: *mut tz_handle, pool_indices: *const u32, params: *const tz_reanalyze_t) -> c_int;
    pub fn tz_reanalyze_read(h: *mut tz_handle, stride: c_int, out_policy: *mut f32, out_ube: *mut f32, out_value: *mut f32, out_n: *mut c_int, out_moves: *mut tz_move_t) -> c_int;
    pub fn tz_profile_begin(h: *mut tz_handle, sample_every: c_int) -> c_int;
    pub fn tz_profile_end(h: *mut tz_handle, out: *mut tz_profile_t) -> c_int;
    pub fn tz_timer_start(h: *mut tz_handle) -> c_int;
    pub fn tz_timer_stop(h: *mut tz_handle, out_ms: *mut f64) -> c_int;
    pub fn tz_tree_simulate_simple(h: *mut tz_handle, beta: f32) -> c_int;
    pub fn tz_tree_simulate_batch(h: *mut tz_handle, beta: f32, batch_size: c_int) -> c_int;
    pub fn tz_tree_descend(h: *mut tz_handle, move_: tz_move_t) -> c_int;
    pub fn tz_tree_principal_variation(h: *mut tz_handle, out_moves: *mut tz_move_t, cap: c_int) -> c_int;
    pub fn tz_trees_simulate_batch(h: *mut tz_handle, mask: *const u8, beta: f32, batch_size: c_int) -> c_int;
    pub fn tz_trees_descend(h: *mut tz_handle, mask: *const u8, moves: *const tz_move_t) -> c_int;
    pub fn tz_trees_principal_variation(h: *mut tz_handle, mask: *const u8, cap: c_int, out_moves: *mut tz_move_t, out_len: *mut c_int) -> c_int;
    pub fn tz_set_weights(h: *mut tz_handle, tensors: *const tz_tensor_t, count: c_int) -> c_int;
    pub fn tz_comm_unique_id(out_id128: *mut c_void) -> c_int;
    pub fn tz_comm_init(h: *mut tz_handle, id128: *const c_void, nranks: c_int, rank: c_int) -> c_int;
    pub fn tz_comm_destroy(h: *mut tz_handle) -> c_int;
    pub fn tz_broadcast_weights(h: *mut tz_handle, tensors: *const tz_tensor_t, count: c_int, res_blocks: c_int, root: c_int) -> c_int;
    pub fn tz_weight_generation(h: *mut tz_handle, out_generation: *mut u64, out_ms: *mut f64) -> c_int;
    pub fn tz_allreduce_sum(h: *mut tz_handle, values: *mut u64, count: c_int) -> c_int;
    pub fn tz_load_model(h: *mut tz_handle, path: *const c_char) -> c_int;
    pub fn tz_load_model_ex(h: *mut tz_handle, path: *const c_char, allow_missing_set: c_int) -> c_int;
    pub fn tz_read_model_file(path: *const c_char, fn_: tz_model_tensor_fn, ctx: *mut c_void) -> c_int;
    pub fn tz_set_network_dtype(h: *mut tz_handle, dtype: c_int) -> c_int;
    pub fn tz_evaluate(h: *mut tz_handle, states: *const tz_state_t, count: c_int, actions: *const tz_move_t, n_actions: *const c_int, stride: c_int, logits: *mut f32, values: *mut f32, variances: *mut f32) -> c_int;
    pub fn tz_set_simhash(h: *mut tz_handle, matrix: *const f32, bitset: *const u8) -> c_int;
    pub fn tz_simhash_indices(h: *mut tz_handle, states: *const tz_state_t, count: c_int, out: *mut u32) -> c_int;
    pub fn tz_set_lcghash(h: *mut tz_handle, init: *const f32, bitset: *const u8) -> c_int;
    pub fn tz_lcghash_indices(h: *mut tz_handle, states: *const tz_state_t, count: c_int, out: *mut u32) -> c_int;
    pub fn tz_update_counts(h: *mut tz_handle, states: *const tz_state_t, count: c_int) -> c_int;
    pub fn tz_read_novelty_set(h: *mut tz_handle, out: *mut u8, cap: usize) -> c_int;
    pub fn tz_encode_planes(h: *mut tz_handle, states: *const tz_state_t, count: c_int, out: *mut f32) -> c_int;
    pub fn tz_debug_layer_limit(h: *mut tz_handle, limit: c_int) -> c_int;
    pub fn tz_debug_activations(h: *mut tz_handle, which: c_int, count: c_int, out: *mut f32) -> c_int;
    pub fn tz_debug_schedule(count: c_int, count_max: c_int, board_n: c_int, chunk_min_tiles: c_int, layers: c_int, out: *mut c_longlong, out_items: *mut c_int, cap: c_int) -> c_int;
    pub fn tz_debug_network_mode(h: *mut tz_handle, per_layer_launches: c_int, chunk_min_tiles: c_int, drop_progress: c_int) -> c_int;
    pub fn tz_debug_tree_warps(h: *mut tz_handle, warps: c_int) -> c_int;
    pub fn tz_debug_weight_set(h: *mut tz_handle, out: *mut u8, cap: usize, out_size: *mut usize) -> c_int;
    pub fn tz_debug_expf(h: *mut tz_handle, in_: *const f32, count: c_int, out: *mut f32) -> c_int;
    pub fn tz_debug_time_tower(h: *mut tz_handle, count: c_int, reps: c_int, ms_per_conv: *mut f64) -> c_int;
}
