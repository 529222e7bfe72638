// tabq.cu -- the finite-space agents: tabular Q-learning (src/agents/tabular.rs:84-232), UCB1 (src/agents/bandits/ucb.rs) and
// Beta Thompson sampling (src/agents/bandits/thompson_sampling.rs).
//
// The reference update is a strictly sequential fold over the buffer whose bootstrap term reads the
// live table (tabular.rs:160-178), so a single shared table cannot be updated in parallel and stay
// bit-exact.  The data-parallel unit here is the replica: replica r owns table r and folds lane r of
// the trajectory in order -- atomic-free, f64 values and u64 counts bit-identical to the reference
// fold of that lane.  K7: latency-bound (one dependent read-modify-write per step per replica).
#include <cmath>
#include <vector>

#include "handles.cuh"

namespace {

__global__ void __launch_bounds__(128)
    tabq_update_kernel(double *__restrict__ q, unsigned long long *__restrict__ counts, uint64_t R, int S, int A,
                       double discount, const float *__restrict__ obs, const float *__restrict__ next_obs,
                       const uint8_t *__restrict__ action, const float *__restrict__ reward,
                       const uint8_t *__restrict__ succ, uint64_t T, uint64_t E, int F) {
    const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (tid >= R) return;
    double *tq = q + tid * (uint64_t)S * A;
    unsigned long long *tc = counts + tid * (uint64_t)S * A;
    // one table per lane: replica tid folds lane tid; one shared table (R == 1): thread 0 folds every lane in order
    const uint64_t lane_begin = R == E ? tid : 0, lane_end = R == E ? tid + 1 : E;
    for (uint64_t r = lane_begin; r < lane_end; ++r) {
    // finite observation spaces are stored one-hot (index.rs:97-115); recover the index
    auto obs_index = [&](const float *planes, uint64_t t) {
        int idx = 0;
        for (int f = 0; f < F; ++f)
            if (planes[(t * F + f) * E + r] != 0.0f) idx = f;
        return idx;
    };
    int cur = T > 0 ? obs_index(obs, 0) : 0;
    for (uint64_t t = 0; t < T; ++t) {
        const uint8_t sc = succ[t * E + r];
        if (sc == RL_PAD) break;
        // fold_transient (simulation/mod.rs:287-313): Continue borrows the next step's observation
        int nxt = 0;
        bool has_next = false;
        if (sc == RL_CONTINUE) {
            if (t + 1 >= T || succ[(t + 1) * E + r] == RL_PAD) break;  // trailing Continue is skipped
            nxt = obs_index(obs, t + 1);
            has_next = true;
        } else if (sc == RL_INTERRUPT) {
            nxt = obs_index(next_obs, t);
            has_next = true;
        }
        // step_update (tabular.rs:159-179)
        double discounted_next = 0.0;
        if (has_next) {
            double m = tq[nxt * A];
            for (int k = 1; k < A; ++k) m = fmax(m, tq[nxt * A + k]);
            discounted_next = __dmul_rn(m, discount);
        }
        const int idx = cur * A + action[t * E + r];
        const unsigned long long c = tc[idx] + 1ull;
        tc[idx] = c;
        const double value = __dadd_rn((double)reward[t * E + r], discounted_next);
        const double weight = __ddiv_rn(1.0, (double)c);
        double qv = __dmul_rn(tq[idx], __dsub_rn(1.0, weight));
        qv = __dadd_rn(qv, __dmul_rn(weight, value));
        tq[idx] = qv;
        if (sc == RL_CONTINUE) cur = nxt;
        else if (t + 1 < T && succ[(t + 1) * E + r] != RL_PAD) cur = obs_index(obs, t + 1);
    }
    }
}

// BaseUCB1Agent::batch_update (ucb.rs:186-199) = step_update (:143-160) over every stored step, lane after lane.
__global__ void __launch_bounds__(128)
    ucb1_update_kernel(double *__restrict__ mean, unsigned long long *__restrict__ count, unsigned long long *__restrict__ visits,
                       uint64_t R, int S, int A, double shift, double scale, const float *__restrict__ obs,
                       const uint8_t *__restrict__ action, const float *__restrict__ reward, const uint8_t *__restrict__ succ,
                       uint64_t T, uint64_t E, int F) {
    const uint64_t tid = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (tid >= R) return;
    double *tm = mean + tid * (uint64_t)S * A;
    unsigned long long *tc = count + tid * (uint64_t)S * A, *tv = visits + tid * (uint64_t)S;
    const uint64_t lane_begin = R == E ? tid : 0, lane_end = R == E ? tid + 1 : E;
    for (uint64_t r = lane_begin; r < lane_end; ++r)
        for (uint64_t t = 0; t < T; ++t) {
            if (succ[t * E + r] == RL_PAD) break;
            int o = 0;  // finite observation spaces are stored one-hot (index.rs:97-115)
            for (int f = 0; f < F; ++f)
                if (obs[(t * F + f) * E + r] != 0.0f) o = f;
            const int idx = o * A + action[t * E + r];
            const double scaled = __dmul_rn(__dadd_rn((double)reward[t * E + r], shift), scale);
            tv[o] += 1ull;
            const unsigned long long c = tc[idx] + 1ull;
            tc[idx] = c;
            const double m = tm[idx];
            tm[idx] = __dadd_rn(m, __ddiv_rn(__dsub_rn(scaled, m), (double)c));
        }
}

// BaseBetaThompsonSamplingAgent::batch_update (thompson_sampling.rs:166-177) = step_update (:126-136) over every stored
// step: one thread per lane.  The counts are integer increments, so a shared table (R == 1) takes every lane's steps
// through atomics and ends bit-identical to the reference's sequential fold in any order.
__global__ void __launch_bounds__(128)
    bts_update_kernel(unsigned long long *__restrict__ low, unsigned long long *__restrict__ high, uint64_t R, int S, int A,
                      double threshold, const float *__restrict__ obs, const uint8_t *__restrict__ action,
                      const float *__restrict__ reward, const uint8_t *__restrict__ succ, uint64_t T, uint64_t E, int F) {
    const uint64_t r = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= E) return;
    const uint64_t base = R == E ? r * (uint64_t)S * A : 0;
    for (uint64_t t = 0; t < T; ++t) {
        if (succ[t * E + r] == RL_PAD) break;
        int o = 0;  // finite observation spaces are stored one-hot (index.rs:97-115)
        for (int f = 0; f < F; ++f)
            if (obs[(t * F + f) * E + r] != 0.0f) o = f;
        const uint64_t idx = base + (uint64_t)o * A + action[t * E + r];
        atomicAdd((double)reward[t * E + r] > threshold ? &high[idx] : &low[idx], 1ull);
    }
}

}  // namespace

extern "C" {

rl_status rl_bts_create(rl_ctx *ctx, uint64_t num_replicas, int32_t num_observations, int32_t num_actions, double reward_lo,
                        double reward_hi, int32_t num_samples, rl_bts **out) {
    RL_REQUIRE(ctx, ctx && out, "rl_bts_create: NULL argument");
    RL_REQUIRE(ctx, num_replicas > 0 && num_observations > 0 && num_actions > 0, "rl_bts_create: empty table");
    RL_REQUIRE(ctx, num_samples >= 1 && num_samples <= 1024, "rl_bts_create: num_samples must be in 1 .. 1024");
    RL_CUDA(ctx, cudaSetDevice(ctx->device));
    rl_bts *b = new (std::nothrow) rl_bts();
    if (!b) return rl_fail(ctx, RL_ERR_OOM, "rl_bts_create: host allocation failed");
    b->ctx = ctx; b->R = num_replicas; b->S = num_observations; b->A = num_actions; b->num_samples = num_samples;
    b->threshold = (reward_lo + reward_hi) / 2.0;  // thompson_sampling.rs:102-103
    const size_t n = (size_t)num_replicas * num_observations * num_actions;
    cudaError_t e = cudaMalloc((void **)&b->low, n * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMalloc((void **)&b->high, n * sizeof(unsigned long long));
    if (e != cudaSuccess) {
        rl_bts_destroy(b);
        return rl_fail(ctx, RL_ERR_OOM, "rl_bts_create: %s", cudaGetErrorString(e));
    }
    std::vector<unsigned long long> ones(n, 1ull);  // (1, 1) for every observation-action pair (:104-105)
    const rl_status st = rl_bts_set_counts(b, (const uint64_t *)ones.data(), (const uint64_t *)ones.data());
    if (st != RL_OK) {
        rl_bts_destroy(b);
        return st;
    }
    *out = b;
    return RL_OK;
}

rl_status rl_bts_destroy(rl_bts *b) {
    if (!b) return RL_OK;
    cudaSetDevice(b->ctx->device);
    cudaStreamSynchronize(b->ctx->stream);
    cudaFree(b->low); cudaFree(b->high);
    delete b;
    return RL_OK;
}

rl_status rl_bts_update(rl_bts *b, rl_traj *traj) {
    if (!b || !traj) return rl_fail(b ? b->ctx : nullptr, RL_ERR_INVALID_ARG, "rl_bts_update: NULL argument");
    rl_ctx *ctx = b->ctx;
    RL_REQUIRE(ctx, traj->E == b->R || b->R == 1, "rl_bts_update: one replica per lane, or one shared set of counts (num_replicas = 1)");
    RL_REQUIRE(ctx, (int)traj->F == b->S, "rl_bts_update: observation space size mismatch");
    const uint64_t T = traj->used_T ? traj->used_T : traj->T;
    const unsigned block = 128, grid = rl_grid_for(traj->E, block);
    RL_LAUNCH(ctx, bts_update_kernel, grid, block, 0, b->low, b->high, b->R, b->S, b->A, b->threshold, traj->obs, traj->action,
              traj->reward, traj->succ, T, traj->E, (int)traj->F);
    return RL_OK;
}

rl_status rl_bts_get_counts(rl_bts *b, uint64_t *low_host, uint64_t *high_host) {
    if (!b) return rl_fail(nullptr, RL_ERR_INVALID_ARG, "rl_bts_get_counts: NULL argument");
    rl_ctx *ctx = b->ctx;
    const size_t n = (size_t)b->R * b->S * b->A;
    RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (low_host) RL_CUDA(ctx, cudaMemcpy(low_host, b->low, n * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    if (high_host) RL_CUDA(ctx, cudaMemcpy(high_host, b->high, n * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    return RL_OK;
}

rl_status rl_bts_set_counts(rl_bts *b, const uint64_t *low_host, const uint64_t *high_host) {
    if (!b) return rl_fail(nullptr, RL_ERR_INVALID_ARG, "rl_bts_set_counts: NULL argument");
    rl_ctx *ctx = b->ctx;
    const size_t n = (size_t)b->R * b->S * b->A;
    RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (low_host) RL_CUDA(ctx, cudaMemcpy(b->low, low_host, n * sizeof(uint64_t), cudaMemcpyHostToDevice));
    if (high_host) RL_CUDA(ctx, cudaMemcpy(b->high, high_host, n * sizeof(uint64_t), cudaMemcpyHostToDevice));
    return RL_OK;
}

rl_status rl_ucb1_create(rl_ctx *ctx, uint64_t num_replicas, int32_t num_observations, int32_t num_actions, double reward_lo,
                         double reward_hi, double exploration_rate, rl_ucb1 **out) {
    RL_REQUIRE(ctx, ctx && out, "rl_ucb1_create: NULL argument");
    RL_REQUIRE(ctx, num_replicas > 0 && num_observations > 0 && num_actions > 0, "rl_ucb1_create: empty table");
    const double width = reward_hi - reward_lo;
    if (!std::isfinite(width) || !(width > 0.0))  // BuildAgentError::UnboundedReward (ucb.rs:112-117)
        return rl_fail(ctx, RL_ERR_INVALID_ARG, "rl_ucb1_create: UCB1 needs a bounded, non-degenerate reward range");
    RL_CUDA(ctx, cudaSetDevice(ctx->device));
    rl_ucb1 *u = new (std::nothrow) rl_ucb1();
    if (!u) return rl_fail(ctx, RL_ERR_OOM, "rl_ucb1_create: host allocation failed");
    u->ctx = ctx; u->R = num_replicas; u->S = num_observations; u->A = num_actions;
    u->rate = exploration_rate; u->scale = 1.0 / width; u->shift = -reward_lo;
    const size_t n = (size_t)num_replicas * num_observations * num_actions, ns = (size_t)num_replicas * num_observations;
    cudaError_t e = cudaMalloc((void **)&u->mean, n * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc((void **)&u->count, n * sizeof(unsigned long long));
    if (e == cudaSuccess) e = cudaMalloc((void **)&u->visits, ns * sizeof(unsigned long long));
    if (e != cudaSuccess) {
        rl_ucb1_destroy(u);
        return rl_fail(ctx, RL_ERR_OOM, "rl_ucb1_create: %s", cudaGetErrorString(e));
    }
    // one success and one failure for each arm (ucb.rs:125-128)
    std::vector<double> m(n, 0.5);
    std::vector<unsigned long long> c(n, 2ull), v(ns, 2ull * (unsigned long long)num_actions);
    const rl_status st = rl_ucb1_set_tables(u, m.data(), (const uint64_t *)c.data(), (const uint64_t *)v.data());
    if (st != RL_OK) {
        rl_ucb1_destroy(u);
        return st;
    }
    *out = u;
    return RL_OK;
}

rl_status rl_ucb1_destroy(rl_ucb1 *u) {
    if (!u) return RL_OK;
    cudaSetDevice(u->ctx->device);
    cudaStreamSynchronize(u->ctx->stream);
    cudaFree(u->mean); cudaFree(u->count); cudaFree(u->visits);
    delete u;
    return RL_OK;
}

rl_status rl_ucb1_update(rl_ucb1 *u, rl_traj *traj) {
    if (!u || !traj) return rl_fail(u ? u->ctx : nullptr, RL_ERR_INVALID_ARG, "rl_ucb1_update: NULL argument");
    rl_ctx *ctx = u->ctx;
    RL_REQUIRE(ctx, traj->E == u->R || u->R == 1, "rl_ucb1_update: one replica per lane, or one shared set of tables (num_replicas = 1)");
    RL_REQUIRE(ctx, (int)traj->F == u->S, "rl_ucb1_update: observation space size mismatch");
    const uint64_t T = traj->used_T ? traj->used_T : traj->T;
    const unsigned block = 128, grid = rl_grid_for(u->R, block);
    RL_LAUNCH(ctx, ucb1_update_kernel, grid, block, 0, u->mean, u->count, u->visits, u->R, u->S, u->A, u->shift, u->scale, traj->obs,
              traj->action, traj->reward, traj->succ, T, traj->E, (int)traj->F);
    return RL_OK;
}

rl_status rl_ucb1_get_tables(rl_ucb1 *u, double *mean_host, uint64_t *action_count_host, uint64_t *visit_count_host) {
    if (!u) return rl_fail(nullptr, RL_ERR_INVALID_ARG, "rl_ucb1_get_tables: NULL argument");
    rl_ctx *ctx = u->ctx;
    const size_t n = (size_t)u->R * u->S * u->A, ns = (size_t)u->R * u->S;
    RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (mean_host) RL_CUDA(ctx, cudaMemcpy(mean_host, u->mean, n * sizeof(double), cudaMemcpyDeviceToHost));
    if (action_count_host) RL_CUDA(ctx, cudaMemcpy(action_count_host, u->count, n * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    if (visit_count_host) RL_CUDA(ctx, cudaMemcpy(visit_count_host, u->visits, ns * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    return RL_OK;
}

rl_status rl_ucb1_set_tables(rl_ucb1 *u, const double *mean_host, const uint64_t *action_count_host,
                             const uint64_t *visit_count_host) {
    if (!u) return rl_fail(nullptr, RL_ERR_INVALID_ARG, "rl_ucb1_set_tables: NULL argument");
    rl_ctx *ctx = u->ctx;
    const size_t n = (size_t)u->R * u->S * u->A, ns = (size_t)u->R * u->S;
    RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (mean_host) RL_CUDA(ctx, cudaMemcpy(u->mean, mean_host, n * sizeof(double), cudaMemcpyHostToDevice));
    if (action_count_host) RL_CUDA(ctx, cudaMemcpy(u->count, action_count_host, n * sizeof(uint64_t), cudaMemcpyHostToDevice));
    if (visit_count_host) RL_CUDA(ctx, cudaMemcpy(u->visits, visit_count_host, ns * sizeof(uint64_t), cudaMemcpyHostToDevice));
    return RL_OK;
}

rl_status rl_tabq_create(rl_ctx *ctx, uint64_t num_replicas, int32_t num_observations, int32_t num_actions,
                         double discount_factor, rl_tabq **out) {
    RL_REQUIRE(ctx, ctx && out, "rl_tabq_create: NULL argument");
    RL_REQUIRE(ctx, num_replicas > 0 && num_observations > 0 && num_actions > 0, "rl_tabq_create: empty table");
    RL_CUDA(ctx, cudaSetDevice(ctx->device));
    rl_tabq *t = new (std::nothrow) rl_tabq();
    if (!t) return rl_fail(ctx, RL_ERR_OOM, "rl_tabq_create: host allocation failed");
    t->ctx = ctx; t->R = num_replicas; t->S = num_observations; t->A = num_actions; t->discount = discount_factor;
    const size_t n = (size_t)num_replicas * num_observations * num_actions;
    cudaError_t e = cudaMalloc((void **)&t->q, n * sizeof(double));
    if (e == cudaSuccess) e = cudaMalloc((void **)&t->counts, n * sizeof(unsigned long long));
    if (e != cudaSuccess) {
        rl_tabq_destroy(t);
        return rl_fail(ctx, RL_ERR_OOM, "rl_tabq_create: %s", cudaGetErrorString(e));
    }
    // build_agent ignores initial_action_count/value and starts from zeros (tabular.rs:61-78,97-111)
    cudaMemsetAsync(t->q, 0, n * sizeof(double), ctx->stream);
    cudaMemsetAsync(t->counts, 0, n * sizeof(unsigned long long), ctx->stream);
    *out = t;
    return RL_OK;
}

rl_status rl_tabq_destroy(rl_tabq *t) {
    if (!t) return RL_OK;
    cudaSetDevice(t->ctx->device);
    cudaStreamSynchronize(t->ctx->stream);
    cudaFree(t->q); cudaFree(t->counts);
    delete t;
    return RL_OK;
}

rl_status rl_tabq_update(rl_tabq *t, rl_traj *traj) {
    if (!t || !traj) return rl_fail(t ? t->ctx : nullptr, RL_ERR_INVALID_ARG, "rl_tabq_update: NULL argument");
    rl_ctx *ctx = t->ctx;
    RL_REQUIRE(ctx, traj->E == t->R || t->R == 1, "rl_tabq_update: one replica per lane, or one shared table (num_replicas = 1)");
    RL_REQUIRE(ctx, (int)traj->F == t->S, "rl_tabq_update: observation space size mismatch");
    const uint64_t T = traj->used_T ? traj->used_T : traj->T;
    const unsigned block = 128, grid = rl_grid_for(t->R, block);
    RL_LAUNCH(ctx, tabq_update_kernel, grid, block, 0, t->q, t->counts, t->R, t->S, t->A, t->discount, traj->obs,
              traj->next_obs, traj->action, traj->reward, traj->succ, T, traj->E, (int)traj->F);
    return RL_OK;
}

rl_status rl_tabq_get_table(rl_tabq *t, double *q_host, uint64_t *counts_host) {
    if (!t) return rl_fail(nullptr, RL_ERR_INVALID_ARG, "rl_tabq_get_table: NULL argument");
    rl_ctx *ctx = t->ctx;
    const size_t n = (size_t)t->R * t->S * t->A;
    RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (q_host) RL_CUDA(ctx, cudaMemcpy(q_host, t->q, n * sizeof(double), cudaMemcpyDeviceToHost));
    if (counts_host) RL_CUDA(ctx, cudaMemcpy(counts_host, t->counts, n * sizeof(uint64_t), cudaMemcpyDeviceToHost));
    return RL_OK;
}

rl_status rl_tabq_set_table(rl_tabq *t, const double *q_host, const uint64_t *counts_host) {
    if (!t) return rl_fail(nullptr, RL_ERR_INVALID_ARG, "rl_tabq_set_table: NULL argument");
    rl_ctx *ctx = t->ctx;
    const size_t n = (size_t)t->R * t->S * t->A;
    RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (q_host) RL_CUDA(ctx, cudaMemcpy(t->q, q_host, n * sizeof(double), cudaMemcpyHostToDevice));
    if (counts_host) RL_CUDA(ctx, cudaMemcpy(t->counts, counts_host, n * sizeof(uint64_t), cudaMemcpyHostToDevice));
    return RL_OK;
}

}  // extern "C"
