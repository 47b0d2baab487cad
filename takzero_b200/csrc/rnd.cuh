// rnd.cuh -- random network distillation, the local-uncertainty term of the 5x5 network (rnd.cu).
#pragma once
#include "handle.cuh"

struct RndState;
// tensors of `rnd_learning.*`, `rnd_target.*`, `min`, `max` when the model has them; returns TZ_OK (also when it has
// none: the estimator is then switched off), or an error for an incomplete / misshapen set
int rnd_set_weights(tz_handle* h, const char* const* names, const float* const* data, const long long* const* shapes,
                    const int* ndims, int count);
bool rnd_ready(const tz_handle* h);
// normalized_rnd of the queued positions below the device-side count `*count_ptr` (null: all `count_max`) ->
// rnd_uncertainty(h)[slot].  The GEMMs run over `count_max` rows; a slot at or above the count is never loaded, its
// input row is zero and its uncertainty is not written.
int rnd_forward(tz_handle* h, const TzState* states, const int* count_ptr, int count_max);
const float* rnd_uncertainty(const tz_handle* h);
void rnd_free(tz_handle* h);
const char* rnd_last_error();
