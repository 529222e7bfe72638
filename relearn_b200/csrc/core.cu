// core.cu -- context, device memory helpers, status strings.
#include "common.cuh"
#include "noise.cuh"

std::string &rl_tls_error() {
    static thread_local std::string err;
    return err;
}

extern "C" {

uint32_t rl_version(void) { return (RL_VERSION_MAJOR << 16) | RL_VERSION_MINOR; }

int32_t rl_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

const char *rl_status_str(rl_status s) {
    switch (s) {
    case RL_OK: return "ok";
    case RL_ERR_INVALID_ARG: return "invalid argument";
    case RL_ERR_CUDA: return "CUDA error";
    case RL_ERR_UNSUPPORTED: return "unsupported configuration";
    case RL_ERR_OOM: return "out of device memory";
    case RL_ERR_NCCL: return "NCCL error";
    case RL_ERR_BUFFER_FULL: return "history buffer full";
    case RL_STEP_NAN_LOSS: return "optimizer step: NaN loss";
    case RL_STEP_NAN_CONSTRAINT: return "optimizer step: NaN constraint";
    case RL_STEP_LOSS_NOT_IMPROVING: return "optimizer step: loss not improving";
    case RL_STEP_CONSTRAINT_VIOLATED: return "optimizer step: constraint violated";
    default: return "unknown status";
    }
}

const char *rl_last_error(rl_ctx *ctx) { return ctx ? ctx->last_error.c_str() : rl_tls_error().c_str(); }

rl_status rl_ctx_create(int32_t device, void *stream, rl_ctx **out) {
    if (!out) return rl_fail(nullptr, RL_ERR_INVALID_ARG, "rl_ctx_create: out is NULL");
    *out = nullptr;
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess || n == 0) {
        cudaGetLastError();
        return rl_fail(nullptr, RL_ERR_CUDA,
                       "rl_ctx_create: no CUDA device available (%s); relearn_b200 has no CPU fallback",
                       e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
    }
    if (device < 0 || device >= n) return rl_fail(nullptr, RL_ERR_INVALID_ARG, "rl_ctx_create: bad device %d", device);
    rl_ctx *ctx = new (std::nothrow) rl_ctx();
    if (!ctx) return rl_fail(nullptr, RL_ERR_OOM, "rl_ctx_create: host allocation failed");
    ctx->device = device;
    RL_CUDA(ctx, cudaSetDevice(device));
    cudaDeviceProp prop;
    RL_CUDA(ctx, cudaGetDeviceProperties(&prop, device));
    ctx->sm_count = prop.multiProcessorCount;
    ctx->cc_major = prop.major;
    ctx->cc_minor = prop.minor;
    ctx->total_mem = prop.totalGlobalMem;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    if (stream) {
        ctx->stream = (cudaStream_t)stream;
    } else {
        RL_CUDA(ctx, cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
        ctx->owns_stream = true;
    }
    *out = ctx;
    return RL_OK;
}

rl_status rl_ctx_destroy(rl_ctx *ctx) {
    if (!ctx) return RL_OK;
    cudaSetDevice(ctx->device);
    cudaStreamSynchronize(ctx->stream);
    rl_nccl_teardown(ctx);
    if (ctx->scratch) cudaFree(ctx->scratch);
    if (ctx->scratch2) cudaFree(ctx->scratch2);
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    if (ctx->rollout_ticket) cudaFree(ctx->rollout_ticket);
    for (cudaEvent_t ev : ctx->upd_ev)
        if (ev) cudaEventDestroy(ev);
    if (ctx->owns_stream) cudaStreamDestroy(ctx->stream);
    delete ctx;
    return RL_OK;
}

rl_status rl_ctx_synchronize(rl_ctx *ctx) {
    RL_REQUIRE(ctx, ctx, "ctx is NULL");
    RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return RL_OK;
}

uint64_t rl_ctx_launch_count(rl_ctx *ctx) { return ctx ? ctx->launches : 0; }

rl_status rl_ctx_device_info(rl_ctx *ctx, int32_t *sm_count, int32_t *cc_major, int32_t *cc_minor,
                             uint64_t *total_mem_bytes) {
    RL_REQUIRE(ctx, ctx, "ctx is NULL");
    if (sm_count) *sm_count = ctx->sm_count;
    if (cc_major) *cc_major = ctx->cc_major;
    if (cc_minor) *cc_minor = ctx->cc_minor;
    if (total_mem_bytes) *total_mem_bytes = ctx->total_mem;
    return RL_OK;
}

rl_status rl_malloc(rl_ctx *ctx, size_t bytes, void **out_dev) {
    RL_REQUIRE(ctx, ctx && out_dev, "rl_malloc: NULL argument");
    RL_CUDA(ctx, cudaSetDevice(ctx->device));
    RL_CUDA(ctx, cudaMalloc(out_dev, bytes ? bytes : 1));
    return RL_OK;
}

rl_status rl_free(rl_ctx *ctx, void *dev) {
    RL_REQUIRE(ctx, ctx, "ctx is NULL");
    if (dev) {
        RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        RL_CUDA(ctx, cudaFree(dev));
    }
    return RL_OK;
}

rl_status rl_memcpy_h2d(rl_ctx *ctx, void *dst_dev, const void *src_host, size_t bytes) {
    RL_REQUIRE(ctx, ctx && (bytes == 0 || (dst_dev && src_host)), "rl_memcpy_h2d: NULL argument");
    RL_CUDA(ctx, cudaMemcpyAsync(dst_dev, src_host, bytes, cudaMemcpyHostToDevice, ctx->stream));
    RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return RL_OK;
}

rl_status rl_memcpy_d2h(rl_ctx *ctx, void *dst_host, const void *src_dev, size_t bytes) {
    RL_REQUIRE(ctx, ctx && (bytes == 0 || (dst_host && src_dev)), "rl_memcpy_d2h: NULL argument");
    RL_CUDA(ctx, cudaMemcpyAsync(dst_host, src_dev, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    return RL_OK;
}

rl_status rl_malloc_host(rl_ctx *ctx, size_t bytes, void **out_host) {
    RL_REQUIRE(ctx, ctx && out_host, "rl_malloc_host: NULL argument");
    RL_CUDA(ctx, cudaMallocHost(out_host, bytes ? bytes : 1));
    return RL_OK;
}

rl_status rl_free_host(rl_ctx *ctx, void *host) {
    RL_REQUIRE(ctx, ctx, "ctx is NULL");
    if (host) RL_CUDA(ctx, cudaFreeHost(host));
    return RL_OK;
}

rl_status rl_memset(rl_ctx *ctx, void *dst_dev, int32_t value, size_t bytes) {
    RL_REQUIRE(ctx, ctx && (bytes == 0 || dst_dev), "rl_memset: NULL argument");
    RL_CUDA(ctx, cudaMemsetAsync(dst_dev, value, bytes, ctx->stream));
    return RL_OK;
}

uint64_t rl_philox_slot(uint64_t seed, uint64_t lane, uint32_t step, int32_t stream, uint32_t draw) {
    return rl_philox_slot_impl(seed, lane, step, stream, draw);
}

}  // extern "C"

rl_status rl_ctx_scratch(rl_ctx *ctx, size_t bytes, void **out) {
    if (bytes > ctx->scratch_bytes) {
        if (ctx->scratch) {
            RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            RL_CUDA(ctx, cudaFree(ctx->scratch));
            ctx->scratch = nullptr;
            ctx->scratch_bytes = 0;
        }
        size_t want = bytes < (1u << 20) ? (1u << 20) : bytes;
        RL_CUDA(ctx, cudaMalloc(&ctx->scratch, want));
        ctx->scratch_bytes = want;
    }
    *out = ctx->scratch;
    return RL_OK;
}

rl_status rl_ctx_scratch2(rl_ctx *ctx, size_t bytes, void **out) {
    if (bytes > ctx->scratch2_bytes) {
        if (ctx->scratch2) {
            RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            RL_CUDA(ctx, cudaFree(ctx->scratch2));
            ctx->scratch2 = nullptr;
            ctx->scratch2_bytes = 0;
        }
        cudaError_t e = cudaMalloc(&ctx->scratch2, bytes);
        if (e != cudaSuccess) return rl_fail(ctx, RL_ERR_OOM, "scratch of %zu bytes: %s", bytes, cudaGetErrorString(e));
        ctx->scratch2_bytes = bytes;
    }
    *out = ctx->scratch2;
    return RL_OK;
}

rl_status rl_ctx_pinned(rl_ctx *ctx, size_t bytes, void **out) {
    if (bytes > ctx->pinned_bytes) {
        if (ctx->pinned) {
            RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
            RL_CUDA(ctx, cudaFreeHost(ctx->pinned));
            ctx->pinned = nullptr;
            ctx->pinned_bytes = 0;
        }
        size_t want = bytes < 65536 ? 65536 : bytes;
        RL_CUDA(ctx, cudaMallocHost(&ctx->pinned, want));
        ctx->pinned_bytes = want;
    }
    *out = ctx->pinned;
    return RL_OK;
}
