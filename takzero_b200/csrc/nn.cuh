// nn.cuh -- device ResNet agent (nn.cu) as seen by api.cu.
#pragma once
#include "handle.cuh"

bool nn_ready(const tz_handle* h);
void nn_free(tz_handle* h);
const char* nn_last_error();
int nn_set_weights(tz_handle* h, const char* const* names, const float* const* data, const long long* const* shapes,
                   const int* ndims, int count);
int nn_broadcast_weights(tz_handle* h, const char* const* names, const float* const* data, const long long* const* shapes,
                         const int* ndims, int count, int res_blocks, int root);
int nn_generation_ms(tz_handle* h, double* ms, unsigned long long* generation);
int nn_debug_weight_set(tz_handle* h, unsigned char* out, size_t cap, size_t* size);
// k_expand finishes the heads itself when the agent is the device network: refresh the pointers it uses
void nn_bind_search(tz_handle* h);
cudaStream_t nn_collective_stream(tz_handle* h);
// policy / value / uncertainty of the queued leaf positions: legal logits -> d.logits, head features for k_expand
int nn_forward_queue(tz_handle* h);
// the same for `count` host-supplied positions already in d.leaf_state / d.actions / d.n_actions -> d.logits,
// d.value, d.variance
int nn_forward_host(tz_handle* h, int count);
int nn_encode_planes(tz_handle* h, const TzState* states, int count, float* out_f32);
void nn_set_layer_limit(tz_handle* h, int limit);
int nn_debug_read(tz_handle* h, int which, int count, float* out_dev);
int nn_time_tower(tz_handle* h, int count, int reps, double* ms_per_conv);
int nn_set_simhash(tz_handle* h, const float* matrix, const unsigned char* bitset);
int nn_simhash_indices(tz_handle* h, const TzState* states, int count, uint32_t* out_dev);
int nn_debug_schedule(int count, int count_max, int n, int chunk_min_tiles, int layers, long long* out, int* out_items,
                      int cap);
int nn_set_lcghash(tz_handle* h, const float* init, const unsigned char* bitset);
int nn_lcghash_indices(tz_handle* h, const TzState* states, int count, uint32_t* out_dev);
int nn_update_counts(tz_handle* h, const TzState* states_dev, int count, uint32_t* idx_dev);
int nn_read_novelty_set(tz_handle* h, unsigned char* out_host);
// 0 no hash yet, 1 SimHash, 2 LCG hash
int nn_hash_kind(const tz_handle* h);
// tz_update_counts_buffer: the examples of a validated training batch (explicit arrays already on the device)
int nn_update_counts_buffer(tz_handle* h, const TzTargetRing& R, int batch, const unsigned long long* indices,
                            const int* symmetry, int augment, unsigned long long seed, unsigned long long size,
                            unsigned long long first);
// tz_broadcast_novelty_set
int nn_broadcast_novelty_set(tz_handle* h, const unsigned char* bitset, int root);
