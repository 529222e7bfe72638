// steps.cuh -- what every fused rollout (rollout.cu: K2*, gru.cu: K8*) does per lane besides stepping: the
// OnlineStepsSummary sums (simulation/summary.rs:198-216), VecBuffer::end_experience -> finalize_last_episode
// (agents/buffers/mod.rs:237-261), the deterministic reduction of the sums into the caller's summary, and the actor's
// categorical / greedy action choice.  Each kernel keeps its own step loop and stores; the rules and the data format
// live here.  K2q (rollout_ws6.cuh) spells finalize_last_episode out itself: with the helper, ptxas schedules its
// step loops differently.
#pragma once

#include <cstdint>

#include "../../include/relearn_b200.h"

// Statistics of a rollout: raw f64 sums (count, sum, sum of squares) per lane, per block and in total.
enum { ST_STEPS = 0, ST_R, ST_R2, ST_EPS, ST_ER, ST_ER2, ST_EL, ST_EL2, ST_STORED_STEPS, ST_STORED_EPS, ST_COUNT };

// finalize_last_episode for a lane that took `steps` steps, the last two with successor codes succ_last / succ_prev: the
// dangling last step (it continued) is dropped, and the step before it, if it continued too, becomes an Interrupt.
// The caller does the stores the flags ask for.
struct LaneEnd {
    uint32_t len;    // steps stored
    uint32_t flags;  // bit 0: slot len becomes RL_PAD; bit 1: slot len - 1 becomes RL_INTERRUPT and receives next_obs
};                   // (the observation of the dropped step).  Also the lane's lane_flags.

__device__ __forceinline__ LaneEnd finalize_last_episode(uint32_t steps, int succ_last, int succ_prev) {
    LaneEnd end{steps, 0u};
    if (steps > 0 && succ_last == RL_CONTINUE) {
        end.len = steps - 1;
        end.flags = 1u;
        if (end.len > 0 && succ_prev == RL_CONTINUE) end.flags = 3u;
    }
    return end;
}

struct LaneStats {
    double v[ST_COUNT];
    double cur_reward;
    uint32_t cur_len;
    __device__ void init() {
#pragma unroll
        for (int i = 0; i < ST_COUNT; ++i) v[i] = 0.0;
        cur_reward = 0.0;
        cur_len = 0;
    }
    // OnlineStepsSummary::push (summary.rs:198-216)
    __device__ void push(float reward, int succ) {
        const double r = (double)reward;
        v[ST_STEPS] += 1.0; v[ST_R] += r; v[ST_R2] += r * r;
        cur_len += 1;
        cur_reward += r;
        if (succ != RL_CONTINUE) {
            const double L = (double)cur_len;
            v[ST_EPS] += 1.0; v[ST_ER] += cur_reward; v[ST_ER2] += cur_reward * cur_reward;
            v[ST_EL] += L; v[ST_EL2] += L * L;
            cur_reward = 0.0;
            cur_len = 0;
        }
    }
    // what the lane stores: its length, and its episodes (an Interrupt made by finalize_last_episode ends one more)
    __device__ void set_stored(const LaneEnd &end) {
        double eps = v[ST_EPS];
        if (end.flags & 2u) eps += 1.0;
        v[ST_STORED_STEPS] = (double)end.len;
        v[ST_STORED_EPS] = eps;
    }
};

__device__ __forceinline__ double warp_sum(double x) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    return x;
}

// Deterministic block reduction of the per-lane statistics into partials[blockIdx.x][*].  `red` is the caller's shared
// memory, one row per warp of the block (a __shared__ array declared here would be allocated in every kernel that calls
// this, whatever its block size).
__device__ __forceinline__ void block_reduce_stats(const LaneStats &st, bool contributes, double (*red)[ST_COUNT],
                                                   double *partials) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = (blockDim.x + 31) >> 5;
#pragma unroll
    for (int i = 0; i < ST_COUNT; ++i) {
        const double s = warp_sum(contributes ? st.v[i] : 0.0);
        if (lane == 0) red[warp][i] = s;
    }
    __syncthreads();
    if (threadIdx.x < ST_COUNT) {
        double s = 0.0;
        for (int w = 0; w < nwarps; ++w) s += red[w][threadIdx.x];
        partials[(size_t)blockIdx.x * ST_COUNT + threadIdx.x] = s;
    }
}

// Statistic i of the totals from the per-block partials, in a fixed order (deterministic): lane l adds rows l, l + 32, ...
// (independent coalesced-by-row loads, through L2: K2q's last CTA reads rows other CTAs just wrote), then a shuffle tree
// combines the lanes.  Lane 0 publishes the sum.
__device__ __forceinline__ void finalize_stat(const double *partials, int nblocks, int i, int lane, double *out,
                                              double *traj_counts, double *host_out) {
    double s = 0.0;
#pragma unroll 4
    for (int b = lane; b < nblocks; b += 32) s += __ldcg(partials + (size_t)b * ST_COUNT + i);
    s = warp_sum(s);
    if (lane == 0) {
        out[i] = s;
        // the caller's summary: written straight into page-locked host memory (no separate device-to-host copy)
        if (host_out) host_out[i] = s;
        if (i == ST_STORED_STEPS) traj_counts[0] = s;
        if (i == ST_STORED_EPS) traj_counts[1] = s;
    }
}

// Categorical::new + sample (categorical.rs:29-33,52-54) as inverse CDF over exp(log_softmax(z)).
template <int MAXA>
__device__ __forceinline__ uint32_t categorical_sample(const float *z, int A, float u) {
    float m = z[0];
#pragma unroll
    for (int k = 1; k < MAXA; ++k)
        if (k < A) m = fmaxf(m, z[k]);
    float sum = 0.0f;
#pragma unroll
    for (int k = 0; k < MAXA; ++k)
        if (k < A) sum += expf(z[k] - m);
    const float lse = m + logf(sum);
    float c = 0.0f;
    uint32_t a = (uint32_t)(A - 1);
    bool found = false;
#pragma unroll
    for (int k = 0; k < MAXA; ++k)
        if (k < A && !found) {
            c += expf(z[k] - lse);
            if (u < c) { a = (uint32_t)k; found = true; }
        }
    return a;
}

template <int MAXA>
__device__ __forceinline__ uint32_t argmax_first(const float *z, int A) {
    uint32_t best = 0;
    float bv = z[0];
#pragma unroll
    for (int k = 1; k < MAXA; ++k)
        if (k < A && z[k] > bv) { bv = z[k]; best = (uint32_t)k; }
    return best;
}
