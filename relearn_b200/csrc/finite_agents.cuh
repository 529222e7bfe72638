// finite_agents.cuh -- the step update and action choice of the finite-space agents, for one state, as scalar helpers:
// tabular Q-learning (src/agents/tabular.rs) and UCB1 (src/agents/bandits/ucb.rs).  Every operation is rounded on its
// own (no FMA contraction), as in the reference's f64 arithmetic.  The resetting meta agent's rollout (K2m,
// rollout_meta.cuh) calls them.  actor_act (rollout.cu), tabq_update_kernel and ucb1_update_kernel (tabq.cu) spell the
// same operations out on their tables in device memory; they do not call these helpers, so that their code stays as it
// was.
#pragma once

// BaseTabularQLearningAgent::step_update (tabular.rs:159-179) for a step whose successor is Terminate (no bootstrap
// term): count += 1; weight = 1 / count; q *= 1 - weight; q += weight * (reward + 0).  `count` is the count after
// the increment.
__device__ __forceinline__ double tabq_step_update_terminal(double q, double count, double reward) {
    const double value = __dadd_rn(reward, 0.0);
    const double weight = __ddiv_rn(1.0, count);
    const double qv = __dmul_rn(q, __dsub_rn(1.0, weight));
    return __dadd_rn(qv, __dmul_rn(weight, value));
}

// BaseUCB1Agent::step_update (ucb.rs:143-160): the reward scaled to [0, 1] by the reward range (shift = -lo,
// scale = 1 / (hi - lo), :112-123), then the running mean with the count after its increment.
__device__ __forceinline__ double ucb1_scaled_reward(double reward, double shift, double scale) {
    return __dmul_rn(__dadd_rn(reward, shift), scale);
}
__device__ __forceinline__ double ucb1_mean_update(double mean, double count, double scaled) {
    return __dadd_rn(mean, __ddiv_rn(__dsub_rn(scaled, mean), count));
}

// BaseUCB1Actor::act in training mode (ucb.rs:219-231): 2 ln(visits) once per state, then per action
// sqrt(2 ln(visits) / count) * exploration_rate + mean.  The caller keeps the LAST maximal action (argmax_by,
// utils/iter/cmp.rs:58-76).
__device__ __forceinline__ double ucb1_log_squared_visits(double visits) { return __dmul_rn(2.0, log(visits)); }
__device__ __forceinline__ double ucb1_bound(double log_squared_visits, double count, double mean, double rate) {
    return __dadd_rn(__dmul_rn(__dsqrt_rn(__ddiv_rn(log_squared_visits, count)), rate), mean);
}
