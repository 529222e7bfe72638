// common.cuh -- context, error plumbing and launch accounting shared by every translation unit.
#pragma once

#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdint>
#include <cstdio>
#include <cstring>
#include <new>
#include <string>

#include "../../include/relearn_b200.h"

// Peer mailboxes for the fused row-reduction + all-reduce (update.cu reduce_rows_x_kernel): every rank owns one
// mailbox in its own HBM, mapped into every peer of the node through CUDA IPC (NVLink / NVSwitch peer memory).
constexpr int RL_X_MAX_RANKS = 8;     // one node
constexpr int RL_X_BLOCKS = 64;       // 32-column blocks per message set: W <= 2048
constexpr int RL_X_SLOT = 40;         // doubles per (source rank, block): 32 column sums, count, loss, padding
struct rl_xpeer {
    double *data[RL_X_MAX_RANKS];               // data[owner]: [2 parity][world][RL_X_BLOCKS][RL_X_SLOT]
    unsigned long long *flag[RL_X_MAX_RANKS];   // flag[owner]: [2 parity][world][RL_X_BLOCKS] sequence numbers
    int rank, world;
    int *error;                                 // set when a wait timed out (a peer never arrived)
};

struct rl_ctx {
    int device = 0;
    cudaStream_t stream = nullptr;
    bool owns_stream = false;
    int sm_count = 148;
    int cc_major = 0, cc_minor = 0;
    size_t total_mem = 0;
    size_t smem_optin = 0;  // shared memory one block may opt in to (cudaFuncAttributeMaxDynamicSharedMemorySize + static)
    uint64_t launches = 0;
    std::string last_error;
    // NCCL data-parallel group (nccl.cu)
    void *nccl_comm = nullptr;
    int rank = 0, world = 1;
    // peer mailboxes (nccl.cu sets them up after the communicator; x_ok false => NCCL all-reduce)
    bool x_ok = false;
    rl_xpeer x{};
    void *x_local = nullptr;               // this rank's mailbox allocation
    void *x_remote[RL_X_MAX_RANKS] = {};   // IPC mappings of the peers' mailboxes
    unsigned long long x_seq = 0;          // collectives issued so far (identical on every rank)
    // scratch for small reductions (lazily grown)
    void *scratch = nullptr;
    size_t scratch_bytes = 0;
    // second scratch (the planes of the GEMM-form recurrent passes, gru_big.cu: live at the same time as the first)
    void *scratch2 = nullptr;
    size_t scratch2_bytes = 0;
    // pinned host scratch for scalar read-backs
    void *pinned = nullptr;
    size_t pinned_bytes = 0;
    // K2q's count of finished CTAs (rollout.cu): 0 between launches
    unsigned *rollout_ticket = nullptr;
    // timing events of the update entry points (created once, destroyed with the context: no leak on an early return)
    cudaEvent_t upd_ev[2] = {nullptr, nullptr};
};

std::string &rl_tls_error();

inline rl_status rl_fail(rl_ctx *ctx, rl_status st, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    if (ctx) ctx->last_error = buf;
    rl_tls_error() = buf;
    return st;
}

// The thread's last error is cleared on failure, so that a later RL_LAUNCH cannot report this call's error as its own.
#define RL_CUDA(ctx, expr)                                                                          \
    do {                                                                                            \
        cudaError_t _e = (expr);                                                                    \
        if (_e != cudaSuccess) {                                                                    \
            cudaGetLastError();                                                                     \
            return rl_fail((ctx), _e == cudaErrorMemoryAllocation ? RL_ERR_OOM : RL_ERR_CUDA,       \
                           "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
        }                                                                                           \
    } while (0)

#define RL_REQUIRE(ctx, cond, msg)                                                                  \
    do {                                                                                            \
        if (!(cond)) return rl_fail((ctx), RL_ERR_INVALID_ARG, "%s (%s:%d)", msg, __FILE__, __LINE__); \
    } while (0)

#define RL_TRY(expr)                                                                                \
    do {                                                                                            \
        rl_status _s = (expr);                                                                      \
        if (_s != RL_OK) return _s;                                                                 \
    } while (0)

// Every kernel launch goes through this so that rl_ctx_launch_count() is the library's own count.
#define RL_LAUNCH(ctx, kernel, grid, block, smem, ...)                                              \
    do {                                                                                            \
        kernel<<<(grid), (block), (smem), (ctx)->stream>>>(__VA_ARGS__);                            \
        (ctx)->launches += 1;                                                                       \
        cudaError_t _e = cudaGetLastError();                                                        \
        if (_e != cudaSuccess)                                                                      \
            return rl_fail((ctx), RL_ERR_CUDA, "launch of %s failed: %s (%s:%d)", #kernel,          \
                           cudaGetErrorString(_e), __FILE__, __LINE__);                             \
    } while (0)

void rl_nccl_teardown(rl_ctx *ctx);
rl_status rl_allreduce_f64_inplace(rl_ctx *ctx, double *buf_dev, size_t n);
rl_status rl_ctx_scratch(rl_ctx *ctx, size_t bytes, void **out);
rl_status rl_ctx_scratch2(rl_ctx *ctx, size_t bytes, void **out);
rl_status rl_ctx_pinned(rl_ctx *ctx, size_t bytes, void **out);

inline unsigned rl_div_up(uint64_t a, uint64_t b) { return (unsigned)((a + b - 1) / b); }

// Grid for an elementwise pass over n items with `block` threads: enough CTAs to cover n, which the
// hardware schedules in waves of sm_count * resident CTAs.
inline unsigned rl_grid_for(uint64_t n, unsigned block) { return rl_div_up(n ? n : 1, block); }
