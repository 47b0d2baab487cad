// rnd.cu -- random network distillation (RND), the local-uncertainty term of the reference's 5x5 network.
//
// takzero/src/network/net5.rs:120-146 (`rnd`: view -> x / sum(x^2) -> Linear(in, 1024) -> ReLU -> Linear(1024, 1024) ->
// ReLU -> Linear(1024, 512)), :193-211 (`forward_rnd` = sum((learning(x) - target(x))^2), `normalized_rnd` =
// clamp((rnd - min) / (max - min), 0, 1) * MAXIMUM_VARIANCE) and :271-277 (uncertainty = clamp(max(exp(ube), rnd), 0, 4);
// the combine itself is enc::warp_heads).  Six plain GEMMs per pass: these are library GEMMs (cuBLAS, TF32 tensor-op
// math, opened with dlopen like NCCL), 1 % of the FLOPs of a network pass; everything around them is small kernels.
#include <dlfcn.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <mutex>
#include <string>
#include <vector>

#include "planes.cuh"
#include "rnd.cuh"

#define WPB TZ_WARPS_PER_BLOCK
#define RND_HIDDEN 1024
#define RND_OUT 512

// the slice of cublas_v2.h this file uses
typedef struct cublasContext* cublasHandle_t;
enum { CUBLAS_OP_N = 0, CUBLAS_OP_T = 1 };
enum { CUBLAS_TF32_TENSOR_OP_MATH = 3 };
struct CublasApi {
    void* lib = nullptr;
    int (*Create)(cublasHandle_t*) = nullptr;
    int (*Destroy)(cublasHandle_t) = nullptr;
    int (*SetStream)(cublasHandle_t, cudaStream_t) = nullptr;
    int (*SetMathMode)(cublasHandle_t, int) = nullptr;
    int (*Sgemm)(cublasHandle_t, int, int, int, int, int, const float*, const float*, int, const float*, int, const float*,
                 float*, int) = nullptr;
};
static CublasApi g_cublas;

struct RndState {
    int in = 0, max_positions = 0;
    float* w[2][3] = {{nullptr, nullptr, nullptr}, {nullptr, nullptr, nullptr}};  // [learning, target][layer] row-major [out][in]
    float* b[2][3] = {{nullptr, nullptr, nullptr}, {nullptr, nullptr, nullptr}};
    float lo = 0.0f, hi = 1.0f;  // `min`, `max` of the normalization
    float *x = nullptr, *h1 = nullptr, *h2 = nullptr, *out[2] = {nullptr, nullptr}, *unc = nullptr;
    cublasHandle_t blas = nullptr;
    std::vector<void*> allocs;
};

static thread_local char g_rnd_err[256] = "";
const char* rnd_last_error() { return g_rnd_err; }
#define RND_FAIL(code, ...)                                \
    do {                                                   \
        snprintf(g_rnd_err, sizeof(g_rnd_err), __VA_ARGS__); \
        return code;                                       \
    } while (0)

static int load_cublas() {
    static std::mutex once;
    std::lock_guard<std::mutex> lock(once);
    if (g_cublas.lib) return TZ_OK;
    const char* env = getenv("TZ_CUBLAS_LIB");
    void* lib = nullptr;
    for (const char* name : {env, "libcublas.so.12", "libcublas.so"}) {
        if (!name || !*name) continue;
        lib = dlopen(name, RTLD_NOW | RTLD_GLOBAL);
        if (lib) break;
    }
    if (!lib) RND_FAIL(TZ_EINVAL, "libcublas.so.12 not found (set TZ_CUBLAS_LIB): %s", dlerror());
    CublasApi api;
    api.lib = lib;
#define SYM(field, name)                           \
    *(void**)(&api.field) = dlsym(lib, name);      \
    if (!api.field) RND_FAIL(TZ_EINVAL, "%s missing in libcublas", name);
    SYM(Create, "cublasCreate_v2");
    SYM(Destroy, "cublasDestroy_v2");
    SYM(SetStream, "cublasSetStream_v2");
    SYM(SetMathMode, "cublasSetMathMode");
    SYM(Sgemm, "cublasSgemm_v2");
#undef SYM
    g_cublas = api;
    return TZ_OK;
}

bool rnd_ready(const tz_handle* h) { return h->rnd != nullptr; }
const float* rnd_uncertainty(const tz_handle* h) { return h->rnd ? h->rnd->unc : nullptr; }

void rnd_free(tz_handle* h) {
    RndState* s = h->rnd;
    if (!s) return;
    if (s->blas) g_cublas.Destroy(s->blas);
    for (void* p : s->allocs) cudaFree(p);
    delete s;
    h->rnd = nullptr;
}

// One warp per position: the f32 planes (game_repr order = x.view([-1, input_size])) divided by the sum of their squares.
// Slots from the device-side count (count_ptr, null = count_max) up to count_max hold no position: their row is zero,
// so the GEMMs that run over all count_max rows read defined data there.
__global__ void __launch_bounds__(32 * WPB) k_rnd_input(const TzState* states, const int* count_ptr, int count_max, int n,
                                                         int half_komi, float* out) {
    __shared__ TzState s_state[WPB];
    __shared__ float s_planes[WPB][36 * 36];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q = blockIdx.x * WPB + warp;
    if (q >= count_max) return;
    const int total = (2 * (2 * n + 3 + 2) + 2) * n * n;
    if (q >= (count_ptr ? *count_ptr : count_max)) {
        for (int i = lane; i < total; i += 32) out[(size_t)q * total + i] = 0.0f;
        return;
    }
    TzState* st = &s_state[warp];
    warp_load_state(st, &states[q], lane);
    float* x = s_planes[warp];
    warp_fill_planes(x, st, n, half_komi, lane, false);
    float sq = 0.0f;
    for (int i = lane; i < total; i += 32) sq = fmaf(x[i], x[i], sq);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
    for (int i = lane; i < total; i += 32) out[(size_t)q * total + i] = x[i] / sq;
}

__global__ void k_rnd_bias_act(float* y, const float* bias, size_t total, int cols, int relu) {
    const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= total) return;
    const float v = y[i] + bias[i % cols];
    y[i] = relu ? fmaxf(v, 0.0f) : v;
}

// One warp per position: sum((learning - target)^2) over the 512 outputs (the final biases are added here),
// normalized and scaled like `normalized_rnd`
__global__ void __launch_bounds__(32 * WPB) k_rnd_finish(const float* l, const float* t, const float* bl, const float* bt,
                                                          const int* count_ptr, int count_max, float lo, float hi, float* unc) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int q = blockIdx.x * WPB + warp;
    if (q >= (count_ptr ? *count_ptr : count_max)) return;
    float acc = 0.0f;
    for (int j = lane; j < RND_OUT; j += 32) {
        const float d = (l[(size_t)q * RND_OUT + j] + bl[j]) - (t[(size_t)q * RND_OUT + j] + bt[j]);
        acc = fmaf(d, d, acc);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) unc[q] = fminf(fmaxf((acc - lo) / (hi - lo), 0.0f), 1.0f) * 4.0f;
}

int rnd_set_weights(tz_handle* h, const char* const* names, const float* const* data, const long long* const* shapes,
                    const int* ndims, int count) {
    auto find = [&](const std::string& name) -> int {
        for (int i = 0; i < count; i++)
            if (name == names[i]) return i;
        return -1;
    };
    if (find("rnd_learning.input_linear.weight") < 0) {  // a model without the estimator
        rnd_free(h);
        return TZ_OK;
    }
    const int n = h->d.n, in = (2 * (2 * n + 3 + 2) + 2) * n * n;
    static const char* nets[2] = {"rnd_learning", "rnd_target"};
    static const char* layers[3] = {"input_linear", "hidden_linear", "final_linear"};
    const long long dims[3][2] = {{RND_HIDDEN, in}, {RND_HIDDEN, RND_HIDDEN}, {RND_OUT, RND_HIDDEN}};
    int idx_w[2][3], idx_b[2][3];
    for (int a = 0; a < 2; a++)
        for (int l = 0; l < 3; l++) {
            const std::string base = std::string(nets[a]) + "." + layers[l];
            idx_w[a][l] = find(base + ".weight");
            idx_b[a][l] = find(base + ".bias");
            if (idx_w[a][l] < 0 || idx_b[a][l] < 0) RND_FAIL(TZ_EINVAL, "missing tensor %s.weight / .bias", base.c_str());
            const int w = idx_w[a][l], b = idx_b[a][l];
            if (ndims[w] != 2 || shapes[w][0] != dims[l][0] || shapes[w][1] != dims[l][1] || ndims[b] != 1 ||
                shapes[b][0] != dims[l][0])
                RND_FAIL(TZ_EINVAL, "tensor %s.weight / .bias has the wrong shape", base.c_str());
        }
    const int i_min = find("min"), i_max = find("max");
    int rc = load_cublas();
    if (rc) return rc;
    cudaStreamSynchronize(h->stream);
    RndState* s = h->rnd;
    if (!s || s->in != in || s->max_positions != h->d.Q) {
        rnd_free(h);
        s = new RndState();
        h->rnd = s;
        s->in = in;
        s->max_positions = h->d.Q;
        const size_t Q = (size_t)h->d.Q;
        auto dalloc = [&](float** p, size_t floats) {
            if (cudaMalloc((void**)p, floats * sizeof(float)) != cudaSuccess) return false;
            s->allocs.push_back(*p);
            return true;
        };
        bool ok = dalloc(&s->x, Q * in) && dalloc(&s->h1, Q * RND_HIDDEN) && dalloc(&s->h2, Q * RND_HIDDEN) &&
                  dalloc(&s->out[0], Q * RND_OUT) && dalloc(&s->out[1], Q * RND_OUT) && dalloc(&s->unc, Q);
        for (int a = 0; a < 2 && ok; a++)
            for (int l = 0; l < 3 && ok; l++)
                ok = dalloc(&s->w[a][l], (size_t)dims[l][0] * dims[l][1]) && dalloc(&s->b[a][l], (size_t)dims[l][0]);
        if (!ok || g_cublas.Create(&s->blas) != 0) {
            rnd_free(h);
            RND_FAIL(TZ_ENOMEM, "allocating the RND estimator failed");
        }
        g_cublas.SetMathMode(s->blas, CUBLAS_TF32_TENSOR_OP_MATH);
    }
    for (int a = 0; a < 2; a++)
        for (int l = 0; l < 3; l++) {
            cudaMemcpy(s->w[a][l], data[idx_w[a][l]], (size_t)dims[l][0] * dims[l][1] * sizeof(float), cudaMemcpyHostToDevice);
            cudaMemcpy(s->b[a][l], data[idx_b[a][l]], (size_t)dims[l][0] * sizeof(float), cudaMemcpyHostToDevice);
        }
    s->lo = i_min >= 0 ? data[i_min][0] : 0.0f;  // root.var("min", [1], Const(0.0)), ("max", [1], Const(1.0))
    s->hi = i_max >= 0 ? data[i_max][0] : 1.0f;
    return cudaGetLastError() == cudaSuccess ? TZ_OK : TZ_ECUDA;
}

int rnd_forward(tz_handle* h, const TzState* states, const int* count_ptr, int count_max) {
    RndState* s = h->rnd;
    if (!s) return TZ_OK;
    if (count_max > s->max_positions) return TZ_EINVAL;
    const TzDev& d = h->d;
    const int wblocks = (count_max + WPB - 1) / WPB;
    g_cublas.SetStream(s->blas, h->stream);
    k_rnd_input<<<wblocks, 32 * WPB, 0, h->stream>>>(states, count_ptr, count_max, d.n, d.half_komi, s->x);
    const float one = 1.0f, zero = 0.0f;
    for (int a = 0; a < 2; a++) {
        // row-major Y[B][out] = X[B][in] W^T: column-major Y(out x B) = W(in x out)^T X(in x B)
        auto gemm = [&](const float* W, const float* X, float* Y, int out, int in) {
            return g_cublas.Sgemm(s->blas, CUBLAS_OP_T, CUBLAS_OP_N, out, count_max, in, &one, W, in, X, in, &zero, Y, out);
        };
        auto act = [&](float* Y, const float* bias, int cols) {
            const size_t total = (size_t)count_max * cols;
            k_rnd_bias_act<<<(unsigned)((total + 255) / 256), 256, 0, h->stream>>>(Y, bias, total, cols, 1);
        };
        if (gemm(s->w[a][0], s->x, s->h1, RND_HIDDEN, s->in) != 0) return TZ_ECUDA;
        act(s->h1, s->b[a][0], RND_HIDDEN);
        if (gemm(s->w[a][1], s->h1, s->h2, RND_HIDDEN, RND_HIDDEN) != 0) return TZ_ECUDA;
        act(s->h2, s->b[a][1], RND_HIDDEN);
        if (gemm(s->w[a][2], s->h2, s->out[a], RND_OUT, RND_HIDDEN) != 0) return TZ_ECUDA;
    }
    k_rnd_finish<<<wblocks, 32 * WPB, 0, h->stream>>>(s->out[0], s->out[1], s->b[0][2], s->b[1][2], count_ptr, count_max, s->lo,
                                                      s->hi, s->unc);
    h->launches += 12;
    return cudaGetLastError() == cudaSuccess ? TZ_OK : TZ_ECUDA;
}
