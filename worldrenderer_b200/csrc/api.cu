// Context, scratch and status plumbing of libwr_b200 (replaces dr.RasterizeCudaContext /
// dr.RasterizeGLContext, render.py:31-37).
#include <stdio.h>
#include <stdlib.h>

#include "common.cuh"

extern "C" const char *wr_status_string(int status)
{
    switch (status) {
    case WR_OK: return "ok";
    case WR_ERR_INVALID_ARGUMENT: return "invalid argument";
    case WR_ERR_OUT_OF_MEMORY: return "out of device memory";
    case WR_ERR_CUDA: return "CUDA error";
    case WR_ERR_NO_DEVICE: return "no usable CUDA device";
    case WR_ERR_UNSUPPORTED: return "unsupported configuration";
    default: return "unknown status";
    }
}

extern "C" int wr_version(void) { return WR_B200_ABI_VERSION; }

extern "C" const char *wr_ctx_last_error(const wr_ctx *ctx) { return ctx ? ctx->last_error : ""; }

extern "C" uint64_t wr_ctx_scratch_bytes(const wr_ctx *ctx) { return ctx ? (uint64_t)ctx->scratch_bytes : 0; }

int wr_set_cuda_error(wr_ctx *ctx, cudaError_t e, const char *where)
{
    if (ctx) snprintf(ctx->last_error, sizeof(ctx->last_error), "%s: %s", where, cudaGetErrorString(e));
    return e == cudaErrorMemoryAllocation ? WR_ERR_OUT_OF_MEMORY : WR_ERR_CUDA;
}

extern "C" int wr_ctx_create(int device, wr_ctx **out)
{
    if (!out) return WR_ERR_INVALID_ARGUMENT;
    *out = nullptr;
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess || count <= 0) return WR_ERR_NO_DEVICE;
    if (device < 0 || device >= count) return WR_ERR_INVALID_ARGUMENT;
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return WR_ERR_CUDA;
    if (prop.major != 10) return WR_ERR_NO_DEVICE;  // this library carries sm_100a code only
    wr_ctx *ctx = static_cast<wr_ctx *>(calloc(1, sizeof(wr_ctx)));
    if (!ctx) return WR_ERR_OUT_OF_MEMORY;
    ctx->device = device;
    ctx->sm_count = prop.multiProcessorCount;
    *out = ctx;
    return WR_OK;
}

extern "C" int wr_ctx_profile(wr_ctx *ctx, int enable)
{
    if (!ctx) return WR_ERR_INVALID_ARGUMENT;
    cudaSetDevice(ctx->device);
    if (enable && !ctx->marks[0]) {
        for (int i = 0; i <= WR_MAX_STAGES; ++i) {
            cudaError_t e = cudaEventCreate(&ctx->marks[i]);
            if (e != cudaSuccess) return wr_set_cuda_error(ctx, e, "cudaEventCreate");
        }
    }
    ctx->profiling = enable ? 1 : 0;
    ctx->n_marks = 0;
    return WR_OK;
}

extern "C" int wr_ctx_profile_read(wr_ctx *ctx, float *stage_ms, int capacity)
{
    if (!ctx || !ctx->profiling || ctx->n_marks < 2) return 0;
    cudaSetDevice(ctx->device);
    cudaError_t e = cudaEventSynchronize(ctx->marks[ctx->n_marks - 1]);
    if (e != cudaSuccess) return wr_set_cuda_error(ctx, e, "cudaEventSynchronize");
    const int n = ctx->n_marks - 1;
    for (int i = 0; i < n && i < capacity; ++i) {
        float ms = 0.f;
        cudaEventElapsedTime(&ms, ctx->marks[i], ctx->marks[i + 1]);
        stage_ms[i] = ms;
    }
    return n;
}

extern "C" const char *wr_ctx_profile_stage_name(const wr_ctx *ctx, int i)
{
    if (!ctx || i < 0 || i >= ctx->n_marks) return "";
    return ctx->mark_names[i];
}

extern "C" void wr_ctx_destroy(wr_ctx *ctx)
{
    if (!ctx) return;
    if (ctx->marks[0])
        for (int i = 0; i <= WR_MAX_STAGES; ++i) cudaEventDestroy(ctx->marks[i]);
    if (ctx->scratch) {
        cudaSetDevice(ctx->device);
        // The scratch comes from cudaMallocAsync, and cudaFree does not wait for such memory: kernels of this context's
        // last calls may still read it (a context dropped right after a launch).  Wait for them, then free.
        cudaDeviceSynchronize();
        cudaFree(ctx->scratch);
    }
    free(ctx);
}

// Grow-only scratch, stream-ordered: the old block is released with cudaFreeAsync and the new one comes from
// cudaMallocAsync on the caller's stream, so growth neither synchronises the device (cudaFree would) nor races with
// kernels of earlier calls that still read the old block (they precede the free in stream order).  A context is used
// from one stream at a time (include/wr_b200.h).  Growth inside a stream capture is refused: the captured kernels
// would hold pointers into a block the graph does not own -- warm the context up first (RenderGraph does).
int wr_scratch_reserve(wr_ctx *ctx, size_t bytes, cudaStream_t stream)
{
    if (bytes <= ctx->scratch_bytes) return WR_OK;
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(stream, &cap) == cudaSuccess && cap != cudaStreamCaptureStatusNone) {
        snprintf(ctx->last_error, sizeof(ctx->last_error),
                 "scratch would have to grow (%zu -> %zu bytes) inside a stream capture", ctx->scratch_bytes, bytes);
        return WR_ERR_UNSUPPORTED;
    }
    ctx->clean_bytes = 0;
    if (ctx->scratch) {
        cudaError_t fe = cudaFreeAsync(ctx->scratch, stream);
        if (fe != cudaSuccess) {  // cudaFree does not wait for stream-ordered memory: the stream's kernels may read it
            cudaGetLastError();
            cudaStreamSynchronize(stream);
            cudaFree(ctx->scratch);
        }
        ctx->scratch = nullptr;
        ctx->scratch_bytes = 0;
    }
    const size_t want = bytes + bytes / 8;  // headroom so slightly larger calls do not reallocate
    void *p = nullptr;
    cudaError_t e = cudaMallocAsync(&p, want, stream);
    if (e != cudaSuccess) {
        cudaGetLastError();
        e = cudaMallocAsync(&p, bytes, stream);
        if (e != cudaSuccess) return wr_set_cuda_error(ctx, e, "cudaMallocAsync(scratch)");
        ctx->scratch_bytes = bytes;
    } else {
        ctx->scratch_bytes = want;
    }
    ctx->scratch = p;
    return WR_OK;
}
