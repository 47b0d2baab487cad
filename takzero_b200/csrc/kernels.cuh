// kernels.cuh -- launch prototypes of the rules / tree kernels (kernels.cu).
#pragma once
#include "common.cuh"

void launch_select(const TzDev& d, int phase, int halving_i, const float* betas, cudaStream_t st);
void launch_agent_synth(const TzDev& d, cudaStream_t st);
void launch_expand(const TzDev& d, cudaStream_t st);
void launch_gumbel_noise(const TzDev& d, float* out, int stride, unsigned long long seed, unsigned long long counter,
                         cudaStream_t st);
void launch_gumbel_init(const TzDev& d, int k, const float* gumbel, int stride, cudaStream_t st);
void launch_halve(const TzDev& d, const float* betas, float visits, int remaining, cudaStream_t st);
void launch_finalize(const TzDev& d, uint16_t* out_moves, cudaStream_t st);
// k_step on the games with mask[g] != 0 (all: null)
void launch_step(const TzDev& d, const uint16_t* moves, cudaStream_t st, const uint8_t* mask = nullptr);
// search trees (one CTA / warp per tree): tree t is game d.tree_game[t], t < trees.  The forward appends to the
// evaluation queue, whose count must be zero before the first tree of a batch starts; the backward expands the leaves.
void launch_tree_forward(const TzDev& d, int trees, float beta, int batch_size, int max_forwards, int warps,
                         cudaStream_t st);
void launch_tree_backward(const TzDev& d, int trees, int batch_size, int warps, cudaStream_t st);
void launch_tree_pv(const TzDev& d, int trees, uint16_t* out_moves, int cap, int* out_len, cudaStream_t st);
void launch_new_openings(const TzDev& d, const uint8_t* mask, const int* sym, const int* adj, unsigned long long seed,
                         unsigned long long counter, cudaStream_t st);
void launch_set_positions(const TzDev& d, const TzState* states, const uint8_t* mask, cudaStream_t st);
void launch_reset_roots(const TzDev& d, const uint8_t* mask, cudaStream_t st);
void launch_restart(const TzDev& d, const int* sym, const int* adj, unsigned long long seed, unsigned long long counter,
                    int* out_terminal, TzState* fin_start, uint16_t* fin_replay, int* fin_len, cudaStream_t st,
                    int* out_result = nullptr);
// resident self-play training data: one pending record per game (after launch_targets), and after launch_restart
// the finished games' completed targets and replays into the output queue (three launches)
void launch_record(const TzDev& d, const TzRecorder& r, const float* policy, const float* ube, const int* n, int stride,
                   cudaStream_t st);
void launch_emit(const TzDev& d, const TzRecorder& r, const int* terminal, const int* fin_len, const TzState* fin_start,
                 const uint16_t* fin_replay, int weighted_random_plies, int exploration_games, cudaStream_t st);
void launch_root_table(const TzDev& d, int stride, int* out_n, uint16_t* moves, uint32_t* visits, uint32_t* eval_tag,
                       uint32_t* eval_bits, float* logit, float* prob, float* std_dev, cudaStream_t st);
void launch_root_stats(const TzDev& d, uint32_t* out, cudaStream_t st);
void launch_targets(const TzDev& d, float visitations, float beta, int stride, float* out_policy, float* out_ube,
                    int* out_n, uint16_t* out_moves, cudaStream_t st);
void launch_select_actions(const TzDev& d, int weighted_random_plies, uint32_t threshold, float allowed_drop,
                           const unsigned long long* randoms, unsigned long long seed, unsigned long long counter,
                           uint16_t* out_moves, cudaStream_t st);
void launch_rules_probe(const TzDev& d, const TzState* states, int count, int stride, uint16_t* out_moves, int* out_n,
                        int* out_terminal, int* out_result, cudaStream_t st);
void launch_apply_moves(const TzDev& d, TzState* states, const uint16_t* moves, int count, int* out_ok,
                        cudaStream_t st);
void launch_merge_moves(const TzDev& d, int weighted_random_plies, const uint16_t* sampled, uint16_t* moves,
                        cudaStream_t st);
void launch_set_root_priors(const TzDev& d, int stride, const float* prob, const float* logit, cudaStream_t st);
void launch_random_steps(const TzDev& d, const uint8_t* mask, int steps, unsigned long long seed, cudaStream_t st);

void launch_debug_expf(const float* in, int count, float* out, cudaStream_t st);
void launch_gather_positions(const TzDev& d, const TzState* pool, const uint32_t* indices, cudaStream_t st);
void launch_reanalyze_values(const TzDev& d, const uint16_t* selected, float* out_value, cudaStream_t st);
