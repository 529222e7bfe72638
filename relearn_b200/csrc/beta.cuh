// beta.cuh -- the Beta sampler of the Thompson-sampling agent (src/agents/bandits/thompson_sampling.rs:192-205).
//
// The reference draws through rand_distr's Beta, whose bit stream no reference test pins, so the device defines its own
// sampler on its own noise (DESIGN section 5).  The algorithm below is the contract; the test oracle
// (tests/thompson_oracle.py) restates it operation for operation.  All arithmetic is f64 with every operation rounded on
// its own; `log` is the only operation that may differ from the host's.  Every draw is next_u64 on the actor stream, the
// last Philox stream, so a variable number of draws overlaps no env stream.  U(w) = rl_u64_to_f64(w), in [0, 1).
//  - Normal, Marsaglia polar: u = 2U - 1, v = 2U - 1, s = u u + v v; accept 0 < s < 1 with z = u sqrt(-2 log(s) / s).
//    At most 64 tries, then z = 0.
//  - Gamma(a), a >= 1, Marsaglia-Tsang: d = a - 1/3, c = 1 / sqrt(9 d).  A try draws z and sets b = 1 + c z; b <= 0
//    rejects at once (no uniform drawn), otherwise v = b b b and u = U.  Accept when u < 1 - 0.0331 z^4 (squeeze) or when
//    log(u) < 0.5 z^2 + d - d v + d log(v); the result is d v.  At most 64 tries, then d.
//  - Beta(alpha, beta) = X / (X + Y) with X = Gamma(alpha) drawn first, then Y = Gamma(beta).
// The tries are bounded so that exhausted replay words (all zero) still end.
#pragma once

#include "noise.cuh"

template <bool REPLAY>
__device__ __forceinline__ double rl_normal_sample(LaneNoise<REPLAY> &nz) {
    for (int tries = 0; tries < 64; ++tries) {
        const double u = __dsub_rn(__dmul_rn(2.0, rl_u64_to_f64(nz.template next_u64<RL_STREAM_ACTOR>())), 1.0);
        const double v = __dsub_rn(__dmul_rn(2.0, rl_u64_to_f64(nz.template next_u64<RL_STREAM_ACTOR>())), 1.0);
        const double s = __dadd_rn(__dmul_rn(u, u), __dmul_rn(v, v));
        if (s > 0.0 && s < 1.0) return __dmul_rn(u, __dsqrt_rn(__ddiv_rn(__dmul_rn(-2.0, log(s)), s)));
    }
    return 0.0;
}

template <bool REPLAY>
__device__ __forceinline__ double rl_gamma_sample(LaneNoise<REPLAY> &nz, double a) {
    const double d = __dsub_rn(a, 1.0 / 3.0);
    const double c = __ddiv_rn(1.0, __dsqrt_rn(__dmul_rn(9.0, d)));
    for (int tries = 0; tries < 64; ++tries) {
        const double z = rl_normal_sample<REPLAY>(nz);
        const double b = __dadd_rn(1.0, __dmul_rn(c, z));
        if (!(b > 0.0)) continue;
        const double v = __dmul_rn(__dmul_rn(b, b), b);
        const double u = rl_u64_to_f64(nz.template next_u64<RL_STREAM_ACTOR>());
        const double z2 = __dmul_rn(z, z);
        if (u < __dsub_rn(1.0, __dmul_rn(0.0331, __dmul_rn(z2, z2)))) return __dmul_rn(d, v);
        const double rhs = __dadd_rn(__dsub_rn(__dadd_rn(__dmul_rn(0.5, z2), d), __dmul_rn(d, v)), __dmul_rn(d, log(v)));
        if (log(u) < rhs) return __dmul_rn(d, v);
    }
    return d;
}

template <bool REPLAY>
__device__ __forceinline__ double rl_beta_sample(LaneNoise<REPLAY> &nz, double alpha, double beta) {
    const double x = rl_gamma_sample<REPLAY>(nz, alpha);
    const double y = rl_gamma_sample<REPLAY>(nz, beta);
    return __ddiv_rn(x, __dadd_rn(x, y));
}

// BaseBetaThompsonSamplingActor::act in training mode for one action (thompson_sampling.rs:195-202): the sequential
// f64 sum, from 0.0, of num_samples draws of Beta(alpha = high, beta = low).
template <bool REPLAY>
__device__ __forceinline__ double rl_beta_sample_sum(LaneNoise<REPLAY> &nz, double high, double low, int num_samples) {
    double sum = 0.0;
    for (int j = 0; j < num_samples; ++j) sum = __dadd_rn(sum, rl_beta_sample<REPLAY>(nz, high, low));
    return sum;
}
