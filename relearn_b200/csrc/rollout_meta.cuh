// rollout_meta.cuh -- K2m: the resetting meta agent (ResettingMetaAgent, src/agents/meta.rs:16-227) on the bandit meta-env,
// one thread per lane.  Included by rollout.cu after K2a, whose loop it follows step for step (reset / act / store /
// step / LaneStats::push / TakeAlignedSteps cut / finalize_last_episode).
//
// Steps::step calls Actor::initial_state at every episode start (simulation/steps.rs:113-168), an episode of the
// meta-env is one trial, and every rollout starts fresh episodes (train.rs:135).  So the inner agent lives exactly one
// trial inside one launch: its tables are built at each trial start (meta.rs:146-157) and kept in registers -- at most
// MAX_ARMS values and counts and one visit count, indexed by predicated unrolled loops the way BanditMetaEnv keeps its
// means -- and never reach device memory.  Counts fit in 32 bits: a trial has at most 2 + 65535 pulls of an arm
// (episodes_per_trial is 16 bits of the env state), and a u32 converts to the same double as the u64 it stands for.
//
// Per meta step (meta.rs:159-198), read from the env state (the meta observation carries the same bits):
//  1. with a previous step (has_prev), fold it into the inner agent at once: observation 0, action prev_action, reward
//     prev_reward, successor Terminate (every inner bandit episode is one step, so SerialActorAgent's update bound
//     {1, 0} is met after every step, serial.rs:60-76, buffers/mod.rs:94-101);
//  2. at the end of an inner episode (inner_done) reset the inner actor state (nothing, for all four agents) and
//     take action 0 (some_element, index.rs:57-60) without a draw;
//  3. otherwise act with the inner agent in training mode (SerialActorAgent::new, serial.rs:49).
// The last pull of a trial is never folded in: it ends the trial (Interrupt) and the agent is rebuilt.  Every draw
// comes from the lane's actor stream.
#pragma once

#include "finite_agents.cuh"
#include "beta.cuh"

struct MetaInnerArgs {
    double rate;          // tabular: epsilon; UCB1: exploration rate
    double shift, scale;  // UCB1: the reward scaling (ucb.rs:112-123)
    double threshold;     // Thompson sampling: (reward_min + reward_max) / 2 (thompson_sampling.rs:102-103)
    int num_samples;      // Thompson sampling: Beta draws summed per arm
};

template <int INNER>
struct MetaInnerAgent {
    static constexpr int K = BanditMetaEnv::MAX_ARMS;
    double v[K];      // tabular: action values; UCB1: mean scaled reward
    uint32_t c[K];    // selection counts
    uint32_t visits;  // UCB1: visit count of the single inner observation
    uint32_t low[K], high[K];  // Thompson sampling: low / high reward counts (thompson_sampling.rs:91-92)

    // build_agent over the inner env structure; none of the builders draws (tabular.rs:61-77, ucb.rs:49-74, random.rs)
    __device__ __forceinline__ void build(int k) {
        if constexpr (INNER == RL_INNER_TABULAR_Q) {  // BaseTabularQLearningAgent::new: zeros (tabular.rs:97-111)
#pragma unroll
            for (int i = 0; i < K; ++i) { v[i] = 0.0; c[i] = 0u; }
        } else if constexpr (INNER == RL_INNER_UCB1) {  // one success and one failure per arm (ucb.rs:125-128)
#pragma unroll
            for (int i = 0; i < K; ++i) { v[i] = 0.5; c[i] = 2u; }
            visits = 2u * (uint32_t)k;
        } else if constexpr (INNER == RL_INNER_BETA_THOMPSON) {  // (1, 1) per arm (thompson_sampling.rs:104-105)
#pragma unroll
            for (int i = 0; i < K; ++i) { low[i] = 1u; high[i] = 1u; }
        }
    }

    __device__ __forceinline__ void update(uint32_t action, double reward, const MetaInnerArgs &m) {
        if constexpr (INNER == RL_INNER_TABULAR_Q) {  // tabular.rs:159-179, next = Terminate
#pragma unroll
            for (int i = 0; i < K; ++i)
                if ((uint32_t)i == action) {
                    c[i] += 1u;
                    v[i] = tabq_step_update_terminal(v[i], (double)c[i], reward);
                }
        } else if constexpr (INNER == RL_INNER_UCB1) {  // ucb.rs:143-160
            const double scaled = ucb1_scaled_reward(reward, m.shift, m.scale);
            visits += 1u;
#pragma unroll
            for (int i = 0; i < K; ++i)
                if ((uint32_t)i == action) {
                    c[i] += 1u;
                    v[i] = ucb1_mean_update(v[i], (double)c[i], scaled);
                }
        } else if constexpr (INNER == RL_INNER_BETA_THOMPSON) {  // thompson_sampling.rs:126-136: strictly above, in f64
            const bool is_high = reward > m.threshold;
#pragma unroll
            for (int i = 0; i < K; ++i)
                if ((uint32_t)i == action) {
                    if (is_high) high[i] += 1u;
                    else low[i] += 1u;
                }
        }
    }

    template <bool REPLAY>
    __device__ __forceinline__ uint32_t act(LaneNoise<REPLAY> &nz, int k, const MetaInnerArgs &m) const {
        if constexpr (INNER == RL_INNER_RANDOM) {  // random.rs:71-72
            return rl_gen_range<REPLAY, RL_STREAM_ACTOR>(nz, (uint32_t)k);
        } else if constexpr (INNER == RL_INNER_TABULAR_Q) {
            // tabular.rs:222-232: one f64 draw, drawn even when epsilon is 0; otherwise the first maximal value
            if (rl_u64_to_f64(nz.template next_u64<RL_STREAM_ACTOR>()) < m.rate)
                return rl_gen_range<REPLAY, RL_STREAM_ACTOR>(nz, (uint32_t)k);
            uint32_t best = 0;
            double bv = v[0];
#pragma unroll
            for (int i = 1; i < K; ++i)
                if (i < k && v[i] > bv) { bv = v[i]; best = (uint32_t)i; }
            return best;
        } else if constexpr (INNER == RL_INNER_BETA_THOMPSON) {
            // thompson_sampling.rs:192-205 in training mode: per arm in order, the sum of num_samples Beta(high, low)
            // draws (beta.cuh); argmax_by keeps the LAST maximal element.  The counts are read by a predicated select so
            // that the draw loops are not unrolled per arm.
            uint32_t best = 0;
            double bv = 0.0;
            for (int i = 0; i < k; ++i) {
                uint32_t lo = low[0], hi = high[0];
#pragma unroll
                for (int j = 1; j < K; ++j)
                    if (j == i) { lo = low[j]; hi = high[j]; }
                const double u = rl_beta_sample_sum<REPLAY>(nz, (double)hi, (double)lo, m.num_samples);
                if (i == 0 || u >= bv) { bv = u; best = (uint32_t)i; }
            }
            return best;
        } else {  // ucb.rs:219-231; argmax_by keeps the LAST maximal element (utils/iter/cmp.rs:58-76)
            const double lsv = ucb1_log_squared_visits((double)visits);
            uint32_t best = 0;
            double bv = 0.0;
#pragma unroll
            for (int i = 0; i < K; ++i)
                if (i < k) {
                    const double u = ucb1_bound(lsv, (double)c[i], v[i], m.rate);
                    if (i == 0 || u >= bv) { bv = u; best = (uint32_t)i; }
                }
            return best;
        }
    }
};

// Feature f of BanditMetaEnv::observe for the packed state word w (meta.rs:152-163,357-363): computed per feature so
// that the kernel needs no observation array.
__device__ __forceinline__ float meta_obs_feature(uint32_t w, int k, int f) {
    const bool inner_done = (w >> 26) & 1u, has_prev = (w >> 25) & 1u;
    if (f == 0 || f == 3 + k) return inner_done ? 1.0f : 0.0f;
    if (f == 1) return has_prev ? 0.0f : 1.0f;
    if (f == 2 + k) return has_prev ? (float)((w >> 24) & 1u) : 0.0f;
    return (has_prev && (uint32_t)(f - 2) == ((w >> 16) & 0xFFu)) ? 1.0f : 0.0f;
}

__device__ __forceinline__ void store_meta_obs(float *planes, uint64_t t, uint64_t e, uint64_t E, int F, int k, uint32_t w) {
#pragma unroll
    for (int f = 0; f < BanditMetaEnv::MAXF; ++f)
        if (f < F) planes[((uint64_t)t * F + f) * E + e] = meta_obs_feature(w, k, f);
}

template <int INNER, bool REPLAY>
__global__ void __launch_bounds__(128, 1) rollout_meta_kernel(BanditMetaEnv::Params p, RolloutArgs a, MetaInnerArgs m) {
    using EnvT = BanditMetaEnv;
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = e < a.E;
    LaneStats st;
    st.init();
    if (valid) {
        const int F = a.F, k = (int)p.num_arms;
        LaneNoise<REPLAY> nz;
        nz.init(a.noise, a.lane_offset + e, e);
        const uint32_t t0 = a.noise.step_counter;
        EnvT::State s;
        s.w = 0;
        MetaInnerAgent<INNER> agent;
        uint32_t last_w = 0;  // state word of the last step taken: its observation is the dropped one
        uint32_t n = a.min_steps ? a.min_steps + a.slack : 0;  // take_steps.rs:20-31
        uint32_t i = 0;
        int succ_last = RL_TERMINATE, succ_prev = RL_TERMINATE;
        if (n > 0) {  // train.rs:135: every period starts fresh episodes
            nz.set_step(t0);
            EnvT::template reset<REPLAY>(p, s, nz);
            agent.build(k);
        }
        while (n > 0) {
            nz.set_step(t0 + i);
            const uint32_t w = s.w;
            if ((w >> 25) & 1u) agent.update((w >> 16) & 0xFFu, (double)((w >> 24) & 1u), m);
            const uint32_t action = ((w >> 26) & 1u) ? 0u : agent.act(nz, k, m);
            store_meta_obs(a.obs, i, e, a.E, F, k, w);
            last_w = w;
            float r;
            const int sc = EnvT::template step<REPLAY>(p, s, action, nz, r);
            if (sc == RL_INTERRUPT) store_meta_obs(a.next_obs, i, e, a.E, F, k, s.w);
            if (sc != RL_CONTINUE) {  // a new trial: a new env and a new inner agent (meta.rs:146-157)
                nz.set_step(t0 + i + 1);
                EnvT::template reset<REPLAY>(p, s, nz);
                agent.build(k);
            }
            a.action[(uint64_t)i * a.E + e] = (uint8_t)action;
            a.reward[(uint64_t)i * a.E + e] = r;
            a.succ[(uint64_t)i * a.E + e] = (uint8_t)sc;
            st.push(r, sc);
            succ_prev = succ_last;
            succ_last = sc;
            i += 1;
            n -= 1;
            if (sc != RL_CONTINUE && n <= a.slack) n = 0;  // take_steps.rs:83-88
        }
        const LaneEnd end = finalize_last_episode(i, succ_last, succ_prev);
        if (end.flags & 1u) a.succ[(uint64_t)end.len * a.E + e] = RL_PAD;
        if (end.flags & 2u) {
            a.succ[(uint64_t)(end.len - 1) * a.E + e] = RL_INTERRUPT;
            store_meta_obs(a.next_obs, end.len - 1, e, a.E, F, k, last_w);
        }
        a.lane_len[e] = end.len;
        a.lane_flags[e] = (uint8_t)end.flags;
        st.set_stored(end);
        nz.finish(a.noise, e);
    }
    __shared__ double red[4][ST_COUNT];  // one row per warp of the 128-thread block
    block_reduce_stats(st, valid, red, a.partials);
}
