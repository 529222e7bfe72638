// noise.cuh -- the `&mut Prng` arguments of relearn's Environment / Actor traits on the device.
//
// PHILOX (production): counter-based Philox4x32-10 (Salmon et al. SC'11).  The 64-bit word for
// draw d of stream s at step t of global lane e is pair (d & 1) of
//   Philox(key = seed, counter = (e_lo, e_hi, t, s * 64 + d / 2)).
// Results therefore do not depend on the launch geometry or on how lanes are sharded over GPUs.
//
// REPLAY (parity): per-lane streams of u32 words consumed sequentially, the way rand_core's
// BlockRng hands out ChaCha words to the reference (next_u64 = two consecutive u32, low first).
//
// The u32/u64 -> sample conversions restate rand 0.8.5 (call sites cited per function).
#pragma once

#include <cstdint>

enum { RL_STREAM_ENV_STEP = 0, RL_STREAM_ENV_RESET = 1, RL_STREAM_ACTOR = 2 };

__host__ __device__ inline void rl_philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0,
                                                 uint32_t k1, uint32_t out[4]) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        uint64_t p0 = (uint64_t)0xD2511F53u * c0;
        uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
        uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0;
        uint32_t n1 = (uint32_t)p1;
        uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1;
        uint32_t n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u;
        k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// rl_philox4x32_10 with its ten round keys, which depend only on the key, computed once: for a loop that draws many
// blocks under one seed (the same words).
struct RlPhiloxKeys {
    uint32_t k0[10], k1[10];
};
__device__ __forceinline__ RlPhiloxKeys rl_philox_keys(uint64_t seed) {
    RlPhiloxKeys k;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        k.k0[r] = (uint32_t)seed + (uint32_t)r * 0x9E3779B9u;
        k.k1[r] = (uint32_t)(seed >> 32) + (uint32_t)r * 0xBB67AE85u;
    }
    return k;
}
__device__ __forceinline__ void rl_philox4x32_10_keyed(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, const RlPhiloxKeys &k,
                                                       uint32_t out[4]) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0;
        const uint64_t p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k.k0[r];
        const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k.k1[r];
        c0 = n0; c1 = (uint32_t)p1; c2 = n2; c3 = (uint32_t)p0;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

__host__ __device__ inline uint64_t rl_philox_slot_impl(uint64_t seed, uint64_t lane, uint32_t t, int stream,
                                                        uint32_t draw) {
    uint32_t o[4];
    rl_philox4x32_10((uint32_t)lane, (uint32_t)(lane >> 32), t, (uint32_t)stream * 64u + (draw >> 1), (uint32_t)seed,
                     (uint32_t)(seed >> 32), o);
    return (draw & 1u) ? ((uint64_t)o[2] | ((uint64_t)o[3] << 32)) : ((uint64_t)o[0] | ((uint64_t)o[1] << 32));
}

struct NoiseSource {
    int mode;  // rl_noise_mode
    uint64_t seed;
    uint32_t step_counter;  // global step index of the next step (Philox)
    const uint32_t *env_words;
    const uint32_t *actor_words;
    uint64_t words_per_lane;
    uint32_t *env_cursor;    // u32 [E], replay only
    uint32_t *actor_cursor;  // u32 [E], replay only
};

template <bool REPLAY>
struct LaneNoise;

template <>
struct LaneNoise<false> {
    uint64_t seed, lane;
    uint32_t t;
    uint32_t draw[3];
    __device__ void init(const NoiseSource &src, uint64_t lane_global, uint64_t /*lane_local*/) {
        seed = src.seed;
        lane = lane_global;
        t = src.step_counter;
        draw[0] = draw[1] = draw[2] = 0;
    }
    __device__ void set_step(uint32_t step) {
        t = step;
        draw[0] = draw[1] = draw[2] = 0;
    }
    template <int STREAM>
    __device__ uint64_t next_u64() {
        return rl_philox_slot_impl(seed, lane, t, STREAM, draw[STREAM]++);
    }
    template <int STREAM>
    __device__ uint32_t next_u32() {
        return (uint32_t)next_u64<STREAM>();
    }
    __device__ void finish(const NoiseSource &, uint64_t) {}
};

template <>
struct LaneNoise<true> {
    const uint32_t *ew, *aw;
    uint32_t ecur, acur, nwords;
    __device__ void init(const NoiseSource &src, uint64_t /*lane_global*/, uint64_t lane_local) {
        ew = src.env_words ? src.env_words + lane_local * src.words_per_lane : nullptr;
        aw = src.actor_words ? src.actor_words + lane_local * src.words_per_lane : nullptr;
        ecur = src.env_cursor[lane_local];
        acur = src.actor_cursor[lane_local];
        nwords = (uint32_t)src.words_per_lane;
    }
    __device__ void set_step(uint32_t) {}
    template <int STREAM>
    __device__ uint32_t next_u32() {
        if (STREAM == RL_STREAM_ACTOR) {
            uint32_t w = (aw && acur < nwords) ? aw[acur] : 0u;
            acur += 1;
            return w;
        }
        uint32_t w = (ew && ecur < nwords) ? ew[ecur] : 0u;
        ecur += 1;
        return w;
    }
    template <int STREAM>
    __device__ uint64_t next_u64() {
        uint64_t lo = next_u32<STREAM>();
        uint64_t hi = next_u32<STREAM>();
        return lo | (hi << 32);
    }
    __device__ void finish(const NoiseSource &src, uint64_t lane_local) {
        src.env_cursor[lane_local] = ecur;
        src.actor_cursor[lane_local] = acur;
    }
};

// ---- rand 0.8.5 conversions ------------------------------------------------------------------
// Standard f32 = 24 high bits of a u32 (call site: src/envs/chain.rs:91)
__device__ __forceinline__ float rl_u32_to_f32(uint32_t w) { return (float)(w >> 8) * (1.0f / 16777216.0f); }
// Standard f64 = 53 high bits of a u64 (call site: src/agents/tabular.rs:223)
__device__ __forceinline__ double rl_u64_to_f64(uint64_t w) {
    return __dmul_rn((double)(w >> 11), 1.0 / 9007199254740992.0);
}
// UniformFloat<f64>::sample with precomputed (low, scale) (call sites: cartpole.rs:105, bandits.rs:100)
__device__ __forceinline__ double rl_u64_to_uniform(uint64_t w, double low, double scale) {
    double v12 = __longlong_as_double((long long)((w >> 12) | 0x3FF0000000000000ull));
    double v01 = __dsub_rn(v12, 1.0);
    return __dadd_rn(__dmul_rn(v01, scale), low);
}
// Bernoulli::sample with p_int = (p * 2^64) as u64 (call sites: dqn.rs:366, utils/distributions.rs:113-120)
__host__ __device__ inline uint64_t rl_bernoulli_p_int(double p) {
    double scaled = p * 18446744073709551616.0;
    return scaled >= 18446744073709551616.0 ? 0xFFFFFFFFFFFFFFFFull : (uint64_t)scaled;
}
template <bool REPLAY, int STREAM>
__device__ __forceinline__ bool rl_gen_bool(LaneNoise<REPLAY> &nz, double p) {
    if (p == 1.0) return true;  // ALWAYS_TRUE consumes nothing
    return nz.template next_u64<STREAM>() < rl_bernoulli_p_int(p);
}
// UniformInt::<usize>::sample_single, 0..n (call sites: memory.rs:87, tabular.rs:225, index.rs:66)
template <bool REPLAY, int STREAM>
__device__ __forceinline__ uint32_t rl_gen_range(LaneNoise<REPLAY> &nz, uint32_t n) {
    uint64_t range = n;
    uint64_t zone = (range << __clzll((long long)range)) - 1;
    for (int tries = 0; tries < 64; ++tries) {
        uint64_t v = nz.template next_u64<STREAM>();
        uint64_t lo = v * range;
        uint64_t hi = __umul64hi(v, range);
        if (lo <= zone) return (uint32_t)hi;
    }
    return 0;
}
