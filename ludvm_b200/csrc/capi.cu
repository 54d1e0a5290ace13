// capi.cu -- context management, error reporting and the FP64/FP32 FMA-rate microbenchmarks.
#include "common.cuh"

namespace ludvm {

static thread_local char g_err[512] = "";

int set_error(int code, const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    return code;
}

int scratch_reserve(ludvm_ctx *ctx, int slot, size_t bytes, void **out)
{
    Scratch &s = ctx->dev[slot];
    if (s.bytes < bytes) {
        if (s.ptr) {
            CUDA_TRY(cudaStreamSynchronize(ctx->stream));
            CUDA_TRY(cudaFree(s.ptr));
            s.ptr = nullptr;
            s.bytes = 0;
        }
        size_t want = bytes + bytes / 4 + 256;
        cudaError_t e = cudaMalloc(&s.ptr, want);
        if (e != cudaSuccess) {
            cudaGetLastError();
            return set_error(LUDVM_E_NOMEM, "cudaMalloc(%zu) failed: %s", want, cudaGetErrorString(e));
        }
        s.bytes = want;
    }
    *out = s.ptr;
    return LUDVM_OK;
}

int sym_timeout_check(ludvm_ctx *ctx)
{
    if (!ctx->sym_timeout || !*(volatile int *)ctx->sym_timeout) return LUDVM_OK;
    *(volatile int *)ctx->sym_timeout = 0;
    return set_error(LUDVM_E_CUDA, "k_fast_sym: a warp waited too long for the column states of its predecessor and the "
                                   "launch was abandoned; the results of that step are not valid");
}

int stage_in(ludvm_ctx *ctx, std::initializer_list<HostIn> in)
{
    size_t total = 0;
    for (const HostIn &a : in) {
        ARG_CHECK(a.n >= 0 && (a.n == 0 || a.host != nullptr));
        total += (size_t)a.n;
    }
    void *p;
    int rc = scratch_reserve(ctx, SLOT_IN, total * sizeof(double), &p);
    if (rc) return rc;
    double *b = (double *)p;
    for (const HostIn &a : in) {
        *a.dev = a.n ? b : nullptr;
        if (a.n) CUDA_TRY(cudaMemcpyAsync(b, a.host, (size_t)a.n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        b += a.n;
    }
    return LUDVM_OK;
}

int stage_out(ludvm_ctx *ctx, std::initializer_list<HostOut> out)
{
    size_t total = 0;
    for (const HostOut &a : out) total += (size_t)a.n;
    void *p;
    int rc = scratch_reserve(ctx, SLOT_OUT, total * sizeof(double), &p);
    if (rc) return rc;
    double *b = (double *)p;
    for (const HostOut &a : out) {
        *a.dev = b;
        b += a.n;
    }
    return LUDVM_OK;
}

int copy_back(ludvm_ctx *ctx, std::initializer_list<HostOut> out)
{
    for (const HostOut &a : out)
        if (a.n) CUDA_TRY(cudaMemcpyAsync(a.host, *a.dev, (size_t)a.n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return LUDVM_OK;
}

// Register-resident dependent-chain FMA kernels: 8 independent chains per thread, 2048 threads per SM.
template <typename T>
__global__ void __launch_bounds__(256) fma_rate_kernel(T *out, int iters, T a, T b)
{
    T c0 = threadIdx.x, c1 = c0 + 1, c2 = c0 + 2, c3 = c0 + 3, c4 = c0 + 4, c5 = c0 + 5, c6 = c0 + 6, c7 = c0 + 7;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int k = 0; k < 8; k++) {
            c0 = c0 * a + b; c1 = c1 * a + b; c2 = c2 * a + b; c3 = c3 * a + b;
            c4 = c4 * a + b; c5 = c5 * a + b; c6 = c6 * a + b; c7 = c7 * a + b;
        }
    }
    T s = ((c0 + c1) + (c2 + c3)) + ((c4 + c5) + (c6 + c7));
    if (s == (T)123456789) out[0] = s;  // never true for the chosen a, b; keeps the chains alive
}

template <typename T>
static int measure_rate(ludvm_ctx *ctx, double ms_target, double *rate)
{
    ARG_CHECK(ctx && rate);
    DeviceGuard g(ctx->device);
    T *dummy;
    void *p;
    int rc = scratch_reserve(ctx, SLOT_FLAG, 256, &p);
    if (rc) return rc;
    dummy = (T *)p;
    cudaEvent_t e0, e1;
    CUDA_TRY(cudaEventCreate(&e0));
    CUDA_TRY(cudaEventCreate(&e1));
    const int blocks = ctx->sm_count * 8, threads = 256;
    int iters = 2000;
    float ms = 0.f;
    double best = 0.0;
    for (int rep = 0; rep < 6; rep++) {
        CUDA_TRY(cudaEventRecord(e0, ctx->stream));
        fma_rate_kernel<T><<<blocks, threads, 0, ctx->stream>>>(dummy, iters, (T)0.999999, (T)1e-7);
        ctx->launches++;
        CUDA_TRY(cudaEventRecord(e1, ctx->stream));
        CUDA_TRY(cudaEventSynchronize(e1));
        CUDA_TRY(cudaEventElapsedTime(&ms, e0, e1));
        double fmas = (double)blocks * threads * (double)iters * 64.0;
        double r = fmas / (ms * 1e-3);
        if (rep >= 2 && r > best) best = r;          // first reps calibrate the length
        if (ms < ms_target && rep < 2) iters = (int)(iters * (ms_target / (ms > 0.01f ? ms : 0.01f))) + 1;
    }
    cudaEventDestroy(e0);
    cudaEventDestroy(e1);
    CUDA_TRY(cudaGetLastError());
    *rate = best;
    return LUDVM_OK;
}

}  // namespace ludvm

using namespace ludvm;

LUDVM_API int ludvm_abi_version(void) { return LUDVM_B200_ABI_VERSION; }

LUDVM_API const char *ludvm_last_error(void) { return g_err; }

LUDVM_API int ludvm_ctx_create(int device, void *cuda_stream, ludvm_ctx **out)
{
    ARG_CHECK(out != nullptr);
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        return set_error(LUDVM_E_CUDA, "no CUDA device available (%s); libludvm_b200 has no CPU fallback",
                         e != cudaSuccess ? cudaGetErrorString(e) : "device count is 0");
    }
    ARG_CHECK(device >= 0 && device < ndev);
    DeviceGuard g(device);
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major < 10)
        return set_error(LUDVM_E_UNSUPPORTED, "device %d is sm_%d%d; this library is built for sm_100a only", device,
                         prop.major, prop.minor);
    ludvm_ctx *ctx = new ludvm_ctx();
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    if (cuda_stream) {
        ctx->stream = (cudaStream_t)cuda_stream;
        ctx->own_stream = false;
    } else {
        cudaError_t se = cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking);
        if (se != cudaSuccess) {
            delete ctx;
            return set_error(LUDVM_E_CUDA, "cudaStreamCreate failed: %s", cudaGetErrorString(se));
        }
        ctx->own_stream = true;
    }
    {   // keep freed arenas in the device's default memory pool (stream-ordered allocator) instead of returning them
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
            unsigned long long keep = ~0ULL;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep);
        }
        cudaGetLastError();
    }
    *out = ctx;
    return LUDVM_OK;
}

LUDVM_API int ludvm_ctx_destroy(ludvm_ctx *ctx)
{
    if (!ctx) return LUDVM_OK;
    DeviceGuard g(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    for (auto &s : ctx->dev)
        if (s.ptr) cudaFree(s.ptr);
    if (ctx->sym_timeout) cudaFreeHost(ctx->sym_timeout);
    if (ctx->own_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return LUDVM_OK;
}

LUDVM_API int ludvm_ctx_synchronize(ludvm_ctx *ctx)
{
    ARG_CHECK(ctx != nullptr);
    DeviceGuard g(ctx->device);
    CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return sym_timeout_check(ctx);
}

LUDVM_API int ludvm_ctx_launch_count(ludvm_ctx *ctx, long long *out)
{
    ARG_CHECK(ctx && out);
    *out = ctx->launches;
    return LUDVM_OK;
}

LUDVM_API int ludvm_ctx_last_plan(ludvm_ctx *ctx, int32_t out[8])
{
    ARG_CHECK(ctx && out);
    for (int i = 0; i < 8; i++) out[i] = ctx->plan[i];
    if ((ctx->plan[0] == LUDVM_K_EXACT_ROWS || ctx->plan[0] == LUDVM_K_EXACT_TILED) && ctx->plan[5] == 1 && ctx->range_flag) {
        DeviceGuard g(ctx->device);   // which instantiation the kernel took is decided on the device: read the verdict
        int bad = 0;
        CUDA_TRY(cudaMemcpyAsync(&bad, ctx->range_flag, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
        CUDA_TRY(cudaStreamSynchronize(ctx->stream));
        out[7] = bad;
    }
    return LUDVM_OK;
}

LUDVM_API int ludvm_measure_fp64_fma_rate(ludvm_ctx *ctx, double ms_target, double *dfma_per_s)
{
    return measure_rate<double>(ctx, ms_target, dfma_per_s);
}

LUDVM_API int ludvm_measure_fp32_fma_rate(ludvm_ctx *ctx, double ms_target, double *ffma_per_s)
{
    return measure_rate<float>(ctx, ms_target, ffma_per_s);
}
