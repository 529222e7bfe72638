// passes.cuh -- what the full-batch pass kernels of the update share: the traits of a pass mode and the per-sample loss
// algebra between a module's outputs and its output cotangent.  The MLP passes (update.cu: the FP32-pipe twin and
// mlp_pass_any_kernel) and K10's head (gru_big.cu) call sample_loss.  The tensor-core pass (pass_tc.cuh) keeps its own
// two-action closed form, and K9 (gru_update.cu) its own form over arrays indexed by run-time values; both take the traits
// and constants from here.
#pragma once

#include "handles.cuh"

// f32::MIN: the clamp of log-probabilities in the entropy (categorical.rs:62-68) and in KL(p0 || p)
constexpr float F32_LOWEST = -3.402823466e+38f;

// Whether a pass in `mode` back-propagates (writes a gradient or a Fisher-vector product), or only reports the scalars
__host__ __device__ constexpr bool pass_backward(int mode) {
    return mode == RL_PASS_GRAD || mode == RL_PASS_FVP || mode == RL_PASS_VALUE || mode == RL_PASS_QLOSS || mode == RL_PASS_PPO ||
           mode == RL_PASS_REINFORCE;
}

template <int MODE>
struct PassMode {
    static constexpr bool BACKWARD = pass_backward(MODE);
    static constexpr bool FVP = MODE == RL_PASS_FVP;
    static constexpr bool IS_POLICY = MODE != RL_PASS_VALUE && MODE != RL_PASS_QLOSS;  // outputs are logits
    static constexpr bool USES_ACT = MODE != RL_PASS_VALUE;
    static constexpr bool USES_ADV = MODE == RL_PASS_EVAL || MODE == RL_PASS_GRAD || MODE == RL_PASS_PPO || MODE == RL_PASS_REINFORCE;
    static constexpr bool USES_LP0 = MODE == RL_PASS_EVAL || MODE == RL_PASS_GRAD || MODE == RL_PASS_PPO;
    static constexpr bool USES_TARGET = MODE == RL_PASS_VALUE || MODE == RL_PASS_QLOSS;
};

// 1 / (1 + e^-v) with the hardware reciprocal (MUFU.RCP, <= 1 ulp) instead of the ~10-instruction IEEE division:
// 24 of these per step sit on K9's recurrence
__device__ __forceinline__ float sigm(float v) { return __fdividef(1.0f, 1.0f + expf(-v)); }

// d act(pre) / d pre from the pre-activation and the activation's output; relu'(0) = 0 as in libtorch
__device__ __forceinline__ float act_grad(int act, float pre, float out) {
    switch (act) {
    case RL_ACT_RELU: return pre > 0.0f ? 1.0f : 0.0f;
    case RL_ACT_SIGMOID: return out * (1.0f - out);
    case RL_ACT_TANH: return 1.0f - out * out;
    default: return 1.0f;
    }
}

// lp[k] = z[k] - logsumexp(z) over the A <= MAXA outputs; lp[k] = 0 for k >= A
template <int MAXA>
__device__ __forceinline__ void log_softmax(const float *z, int A, float *lp) {
    float m = z[0];
#pragma unroll
    for (int k = 1; k < MAXA; ++k)
        if (k < A) m = fmaxf(m, z[k]);
    float sum = 0.0f;
#pragma unroll
    for (int k = 0; k < MAXA; ++k)
        if (k < A) sum += expf(z[k] - m);
    const float lse = m + logf(sum);
#pragma unroll
    for (int k = 0; k < MAXA; ++k) lp[k] = k < A ? z[k] - lse : 0.0f;
}

struct SampleLoss {
    float loss, kl, entropy;
};

// One sample's loss, KL and entropy terms and its output cotangent dz[0 .. MAXA) (zero beyond A and where the loss has
// no gradient), from the module's outputs z (FVP: and their tangent zd along the direction).  A <= MAXA is the output
// count (A == MAXA folds every bound); act, adv and tgt are the sample's action, advantage and target; clip = (1 - eps,
// 1 + eps) of PPO; lp0_at(k) returns the behaviour log-probability of action k < A from wherever the kernel keeps it
// (k is the taken action once, else a compile-time index).  lp[] receives the log-probabilities (what STATS stores as
// logp0).  Every loop runs over MAXA with k < A as a predicate and the taken action's log-probability is found by a
// search, so that the per-sample arrays stay in registers.
template <int MODE, int MAXA, class Lp0>
__device__ __forceinline__ SampleLoss sample_loss(const float *z, const float *zd, int A, int act, float adv, float tgt, float2 clip,
                                                  Lp0 lp0_at, float *lp, float *dz) {
    using M = PassMode<MODE>;
    SampleLoss r{0.0f, 0.0f, 0.0f};
#pragma unroll
    for (int k = 0; k < MAXA; ++k) dz[k] = 0.0f;
    if (M::IS_POLICY) {
        float p[MAXA];
        log_softmax<MAXA>(z, A, lp);
#pragma unroll
        for (int k = 0; k < MAXA; ++k) p[k] = k < A ? expf(lp[k]) : 0.0f;
        float lpa = lp[0];  // of the taken action
#pragma unroll
        for (int k = 1; k < MAXA; ++k)
            if (k == act) lpa = lp[k];
        if (MODE == RL_PASS_STATS) {
            // trpo.rs:112-122: log-probs of the behaviour policy and its entropy (categorical.rs:62-68)
#pragma unroll
            for (int k = 0; k < MAXA; ++k)
                if (k < A) r.entropy -= fmaxf(lp[k], F32_LOWEST) * p[k];
        }
        if (M::USES_LP0) {
            const float ratio = expf(lpa - lp0_at(act));
            if (MODE == RL_PASS_PPO) {
                // ppo.rs:124-138: -mean(min(ratio * adv, clip(ratio, 1 - eps, 1 + eps) * adv)).  Backward as libtorch:
                // clamp passes the gradient on [lo, hi] (inclusive), minimum splits it on ties, so d/d ratio = adv when the
                // ratio is inside the clip range or the unclipped term is the smaller.
                const float clipped = fminf(fmaxf(ratio, clip.x), clip.y);
                const float t1 = ratio * adv, t2 = clipped * adv;
                r.loss = -fminf(t1, t2);
                const bool inside = ratio >= clip.x && ratio <= clip.y;
                const float g = (inside || t1 < t2) ? -t1 : 0.0f;
#pragma unroll
                for (int k = 0; k < MAXA; ++k)
                    if (k < A) dz[k] = g * ((act == k ? 1.0f : 0.0f) - p[k]);
            } else {
                // trpo.rs:129-144: ratio = exp(logp - logp0); loss = -mean(ratio * adv); KL(p0 || p)
                r.loss = -(ratio * adv);
#pragma unroll
                for (int k = 0; k < MAXA; ++k)
                    if (k < A) {
                        const float lp0k = lp0_at(k);
                        r.kl += fmaxf(lp0k - lp[k], F32_LOWEST) * expf(lp0k);
                    }
                if (MODE == RL_PASS_GRAD) {
#pragma unroll
                    for (int k = 0; k < MAXA; ++k)
                        if (k < A) dz[k] = r.loss * ((act == k ? 1.0f : 0.0f) - p[k]);
                }
            }
        }
        if (MODE == RL_PASS_REINFORCE) {
            // reinforce.rs:72-79: -(log_probs * advantages).mean(); the entropy of the current policy is logged
            r.loss = -(lpa * adv);
#pragma unroll
            for (int k = 0; k < MAXA; ++k)
                if (k < A) {
                    r.entropy -= fmaxf(lp[k], F32_LOWEST) * p[k];
                    dz[k] = -adv * ((act == k ? 1.0f : 0.0f) - p[k]);
                }
        }
        if (M::FVP) {
            // u = (diag p - p p^T) zdot
            float pd = 0.0f;
#pragma unroll
            for (int k = 0; k < MAXA; ++k)
                if (k < A) pd = fmaf(p[k], zd[k], pd);
#pragma unroll
            for (int k = 0; k < MAXA; ++k)
                if (k < A) dz[k] = p[k] * (zd[k] - pd);
        }
    } else if (MODE == RL_PASS_QLOSS) {
        // dqn.rs:316-326: mse(Q(obs).gather(action), targets); only the taken action's output has a gradient
        float q = z[0];
#pragma unroll
        for (int k = 1; k < MAXA; ++k)
            if (k == act) q = z[k];
        const float diff = q - tgt;
        r.loss = diff * diff;
#pragma unroll
        for (int k = 0; k < MAXA; ++k)
            if (k == act && k < A) dz[k] = 2.0f * diff;
    } else {
        // opt.rs:109-115: mse_loss(V(obs), targets, Mean)
        const float diff = z[0] - tgt;
        r.loss = diff * diff;
        dz[0] = 2.0f * diff;
    }
    return r;
}
