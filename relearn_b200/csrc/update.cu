// update.cu -- the on-policy update: TRPO policy step and Adam critic step.
//
// Reference: Trpo::update (src/torch/agents/policies/trpo.rs:97-164),
// ConjugateGradientOptimizer (src/torch/optimizers/conjugate_gradient.rs:115-403),
// ValuesOpt::update (src/torch/agents/critics/opt.rs:100-127), n_backward_steps
// (src/torch/agents/mod.rs:35-72), COptimizer/Adam (src/torch/optimizers/coptimizer.rs:13-27).
//
// The reference runs ~29 full-batch libtorch passes with autograd (first and second order) and a
// host sync per CG iteration and per line-search try.  Here every pass over the batch is one fused
// kernel (K5/K6) that computes forward, the per-sample softmax algebra and the analytic backward /
// Fisher-vector product, and every piece of P-vector algebra (CG recurrences, step size, line-search
// bookkeeping, Adam) is a single-CTA kernel driven by device-side flags, so the whole update is
// enqueued without a host round trip.
//
// Three kernels run the passes (launch_pass picks one).  Each writes one f64 partial row per CTA; rows
// are summed in a fixed order, so the result is deterministic and independent of scheduling.
//   mlp_pass_tc_kernel<A, MODE> (pass_tc.cuh): the reference's default networks, the 5 -> 128 -> 1
//     critic and the 5 -> 128 -> 2 policy / action-value network, on the tensor cores;
//   mlp_pass_kernel: the same networks on the FP32 pipe, the cross-check of the tensor-core kernel
//     (RL_PASS_KERNEL=ffma or rl_pass_kernel_select(RL_PASS_KERNEL_FFMA));
//   mlp_pass_any_kernel<MODE>: every other supported module, on the FP32 pipe.
//
// Exactness: the Hessian of mean KL(p0 || p_theta) at theta0 equals the Fisher matrix
// mean J^T (diag p - p p^T) J (the first-order term vanishes because p = p0 there), so the analytic
// Fisher-vector product is the reference's double-backward Hessian-vector product.
#include "passes.cuh"

#include <cmath>
#include <cstdlib>
#include <vector>

namespace {

enum { SC_LOSS = 0, SC_KL = 1, SC_ENTROPY = 2, SC_COUNT = 3, NSCALAR = 4 };
constexpr int PASS_THREADS = 256;
constexpr int FLUSH_TILES = 4;

struct PassArgs {
    const float *obs;
    const uint8_t *action, *succ;
    uint64_t T, E;
    const float *theta, *vec;
    const float *adv;
    float *logp0;         // f32 [T*E][2]
    const float *target;  // f32 [T*E]
    double *partials;     // f64 [gridDim.x][P + NSCALAR]
    const int *skip_flag;
    float clip_lo, clip_hi;  // RL_PASS_PPO: 1 -+ clip_distance as f32 (ppo.rs:131-132)
};

// Reduce v[0..CH-1] across the 32 lanes (CH = 8 or 4); afterwards every lane of group g holds the
// complete sum of element g, where groups are 32/CH consecutive lanes.  CH=8: 9 shuffles, CH=4: 6.
template <int CH>
__device__ __forceinline__ float reduce_scatter(float *v, int lane) {
    const bool b4 = lane & 16, b3 = lane & 8, b2 = lane & 4;
    if (CH == 8) {
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float send = b4 ? v[i] : v[i + 4], keep = b4 ? v[i + 4] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
        }
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const float send = b3 ? v[i] : v[i + 2], keep = b3 ? v[i + 2] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
        }
        const float send = b2 ? v[0] : v[1], keep = b2 ? v[1] : v[0];
        v[0] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
    } else {
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const float send = b4 ? v[i] : v[i + 2], keep = b4 ? v[i + 2] : v[i];
            v[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
        }
        const float send = b3 ? v[0] : v[1], keep = b3 ? v[1] : v[0];
        v[0] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
        v[0] += __shfl_xor_sync(0xffffffffu, v[0], 4);
    }
    v[0] += __shfl_xor_sync(0xffffffffu, v[0], 2);
    v[0] += __shfl_xor_sync(0xffffffffu, v[0], 1);
    return v[0];
}

__device__ __forceinline__ double warp_sum_f64(double x) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    return x;
}

// Packed FP32x2 helpers (Blackwell FFMA2/FADD2/FMUL2: one issue slot, two FMAs)
__device__ __forceinline__ float2 f2(float a, float b) { return make_float2(a, b); }
__device__ __forceinline__ float2 dup2(float a) { return make_float2(a, a); }

// mlp_pass_kernel<F, A, UPL, MODE, CH, MINB>: one warp owns a tile of 32 samples; lane l owns hidden units
// {l + 32u : u < UPL} (H = 32 * UPL) with their weights in registers.  Forward computes each lane's
// partial logits for 8 samples at a time and combines them with a shuffle reduce-scatter; the lane
// that loaded sample s does that sample's softmax / loss / KL algebra; the backward sweep re-derives
// the hidden activations (cheaper than staging them through shared memory) and accumulates this
// lane's slice of the parameter gradient in f32 registers, flushed to per-warp f64 totals in shared
// memory every few tiles.
//
// It stays as the FP32 cross-check of the default networks because mlp_pass_any_kernel is not accurate enough
// there: on the saturated two-action policy (logits up to |z| ~ 270) its gradient is 1.1e-4 from f64, against
// 4e-5 for this kernel and a 1e-4 bound (tests/test_gpu_update.py, test_policy_pass_large_logits_and_padding).
template <int F, int A, int UPL, int MODE, int CH, int MINB>
__global__ void __launch_bounds__(PASS_THREADS, MINB) mlp_pass_kernel(PassArgs a) {
    static_assert(UPL % 2 == 0, "hidden units are processed in pairs (FFMA2)");
    constexpr int GROUP = 32 / CH;  // lanes that end up holding the same sample's logits
    constexpr int H = 32 * UPL;
    constexpr int NP = UPL / 2;     // unit pairs per lane: pair q = units (lane + 64 q, lane + 64 q + 32)
    constexpr int P = H * F + H + A * H + A;
    constexpr int W = P + NSCALAR;
    constexpr int XS = 12;          // floats per staged sample: F duplicated pairs (x, x), padded to 3 x float4
    static_assert(2 * F <= XS, "sample stage too small");
    using M = PassMode<MODE>;
    constexpr bool BACKWARD = M::BACKWARD, FVP = M::FVP;
    if (a.skip_flag && *a.skip_flag) return;

    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
    // per-warp regions: f64 totals [P], x tile [32][XS]
    double *tot_all = reinterpret_cast<double *>(smem_raw);
    double *tot = tot_all + (size_t)warp * P;
    float *xs_all = reinterpret_cast<float *>(tot_all + (size_t)nwarps * P);
    float *xs = xs_all + (size_t)warp * 32 * XS;
    if (BACKWARD)
        for (int i = lane; i < P; i += 32) tot[i] = 0.0;

    // this lane's slice of the parameters, as unit pairs (.x = unit lane + 64 q, .y = that + 32)
    const float *tw1 = a.theta, *tb1 = tw1 + H * F, *tw2 = tb1 + H, *tb2 = tw2 + A * H;
    float2 w1[NP][F], b1[NP], w2[A][NP];
    float b2[A];
#pragma unroll
    for (int q = 0; q < NP; ++q) {
        const int j0 = lane + 64 * q, j1 = j0 + 32;
#pragma unroll
        for (int f = 0; f < F; ++f) w1[q][f] = f2(tw1[j0 * F + f], tw1[j1 * F + f]);
        b1[q] = f2(tb1[j0], tb1[j1]);
#pragma unroll
        for (int k = 0; k < A; ++k) w2[k][q] = f2(tw2[k * H + j0], tw2[k * H + j1]);
    }
#pragma unroll
    for (int k = 0; k < A; ++k) b2[k] = tb2[k];
    // FVP direction slice
    float2 vw1[FVP ? NP : 1][F], vb1[FVP ? NP : 1], vw2[A][FVP ? NP : 1];
    float vb2[A];
    if (FVP) {
        const float *pw1 = a.vec, *pb1 = pw1 + H * F, *pw2 = pb1 + H, *pb2 = pw2 + A * H;
#pragma unroll
        for (int q = 0; q < NP; ++q) {
            const int j0 = lane + 64 * q, j1 = j0 + 32;
#pragma unroll
            for (int f = 0; f < F; ++f) vw1[q][f] = f2(pw1[j0 * F + f], pw1[j1 * F + f]);
            vb1[q] = f2(pb1[j0], pb1[j1]);
#pragma unroll
            for (int k = 0; k < A; ++k) vw2[k][q] = f2(pw2[k * H + j0], pw2[k * H + j1]);
        }
#pragma unroll
        for (int k = 0; k < A; ++k) vb2[k] = pb2[k];
    }
    // gradient accumulators (f32 pairs, flushed to f64)
    float2 gw1[BACKWARD ? NP : 1][F], gb1[BACKWARD ? NP : 1], gw2[A][BACKWARD ? NP : 1];
    if (BACKWARD) {
#pragma unroll
        for (int q = 0; q < NP; ++q) {
#pragma unroll
            for (int f = 0; f < F; ++f) gw1[q][f] = f2(0.0f, 0.0f);
            gb1[q] = f2(0.0f, 0.0f);
#pragma unroll
            for (int k = 0; k < A; ++k) gw2[k][q] = f2(0.0f, 0.0f);
        }
    }
    double gb2[A], sc[NSCALAR];
#pragma unroll
    for (int k = 0; k < A; ++k) gb2[k] = 0.0;
#pragma unroll
    for (int k = 0; k < NSCALAR; ++k) sc[k] = 0.0;

    auto flush = [&]() {
        if (!BACKWARD) return;
#pragma unroll
        for (int q = 0; q < NP; ++q) {
            const int j0 = lane + 64 * q, j1 = j0 + 32;
#pragma unroll
            for (int f = 0; f < F; ++f) {
                tot[j0 * F + f] += (double)gw1[q][f].x;
                tot[j1 * F + f] += (double)gw1[q][f].y;
                gw1[q][f] = f2(0.0f, 0.0f);
            }
            tot[H * F + j0] += (double)gb1[q].x;
            tot[H * F + j1] += (double)gb1[q].y;
            gb1[q] = f2(0.0f, 0.0f);
#pragma unroll
            for (int k = 0; k < A; ++k) {
                tot[H * F + H + k * H + j0] += (double)gw2[k][q].x;
                tot[H * F + H + k * H + j1] += (double)gw2[k][q].y;
                gw2[k][q] = f2(0.0f, 0.0f);
            }
        }
    };

    const uint64_t TE = a.T * a.E;
    const uint64_t ntiles = (TE + 31) / 32;
    const uint64_t warp_global = (uint64_t)blockIdx.x * nwarps + warp, total_warps = (uint64_t)gridDim.x * nwarps;
    const int quad_sample = lane / GROUP;  // sample (within a chunk) whose reduced logits this lane receives
    const bool quad_leader = (lane % GROUP) == 0;
    int since_flush = 0;
    // Software pipeline: the global loads of the next tile are in flight while this tile is computed.
    struct Staged {
        float x[F];
        float adv, tgt, lp0a, lp0b;
        int act;
        bool valid;
    };
    // All loads of a tile are issued together: the observation / target / advantage loads do not wait for the
    // successor code (one memory latency per tile instead of two); slots that turn out to be padding are zeroed.
    auto load_tile = [&](uint64_t tile, Staged &st) {
        const uint64_t n = tile * 32 + lane;
        const bool in_range = tile < ntiles && n < TE;
        const uint64_t t = in_range ? n / a.E : 0, e = in_range ? n - t * a.E : 0;
        const uint8_t sc_code = in_range ? __ldg(a.succ + n) : (uint8_t)RL_PAD;
        float x[F];
#pragma unroll
        for (int f = 0; f < F; ++f) x[f] = in_range ? __ldg(a.obs + (t * F + f) * a.E + e) : 0.0f;
        const int act = (M::USES_ACT && in_range) ? (int)__ldg(a.action + n) : 0;
        const float adv = (M::USES_ADV && in_range) ? __ldg(a.adv + n) : 0.0f;
        const float tgt = (M::USES_TARGET && in_range) ? __ldg(a.target + n) : 0.0f;
        float2 l = make_float2(0.0f, 0.0f);
        if (M::USES_LP0 && in_range) l = __ldg(reinterpret_cast<const float2 *>(a.logp0) + n);
        st.valid = sc_code != RL_PAD;
#pragma unroll
        for (int f = 0; f < F; ++f) st.x[f] = st.valid ? x[f] : 0.0f;
        st.act = st.valid ? act : 0;
        st.adv = st.valid ? adv : 0.0f;
        st.tgt = st.valid ? tgt : 0.0f;
        st.lp0a = st.valid ? l.x : 0.0f;
        st.lp0b = st.valid ? l.y : 0.0f;
    };
    Staged nxt;
    load_tile(warp_global, nxt);
    for (uint64_t tile = warp_global; tile < ntiles; tile += total_warps) {
        // ---- stage this lane's sample: duplicated feature pairs to shared memory, scalars in registers ----
        const Staged cur = nxt;
        load_tile(tile + total_warps, nxt);
        const bool valid = cur.valid;
        float xv[XS];
#pragma unroll
        for (int i = 0; i < XS; ++i) xv[i] = (i / 2) < F ? cur.x[(i / 2) < F ? (i / 2) : 0] : 0.0f;
        __syncwarp();
#pragma unroll
        for (int i = 0; i < XS / 4; ++i)
            reinterpret_cast<float4 *>(xs)[lane * (XS / 4) + i] = make_float4(xv[4 * i], xv[4 * i + 1], xv[4 * i + 2], xv[4 * i + 3]);
        const int my_act = cur.act;
        const float my_adv = cur.adv, my_tgt = cur.tgt;
        const float my_lp0[2] = {cur.lp0a, cur.lp0b};
        const unsigned valid_mask = __ballot_sync(0xffffffffu, valid);
        __syncwarp();

#pragma unroll 1
        for (int c = 0; c < 32 / CH; ++c) {
            // ---- forward for samples CH*c .. CH*c+CH-1: this lane's partial logits, activations kept ----
            float2 hid[CH][NP];  // relu(pre); hid > 0 <=> pre > 0
            float pz[A][CH], pzd[FVP ? A : 1][CH];
#pragma unroll
            for (int i = 0; i < CH; ++i) {
                float2 x[XS / 2];
#pragma unroll
                for (int v = 0; v < XS / 4; ++v) {
                    const float4 t4 = reinterpret_cast<const float4 *>(xs)[(c * CH + i) * (XS / 4) + v];
                    x[2 * v] = f2(t4.x, t4.y);
                    x[2 * v + 1] = f2(t4.z, t4.w);
                }
                float2 acc[A], accd[FVP ? A : 1];
#pragma unroll
                for (int k = 0; k < A; ++k) {
                    acc[k] = f2(0.0f, 0.0f);
                    if (FVP) accd[k] = f2(0.0f, 0.0f);
                }
#pragma unroll
                for (int q = 0; q < NP; ++q) {
                    float2 p_ = b1[q];
#pragma unroll
                    for (int f = 0; f < F; ++f) p_ = __ffma2_rn(w1[q][f], x[f], p_);
                    const float2 h = f2(fmaxf(p_.x, 0.0f), fmaxf(p_.y, 0.0f));
                    hid[i][q] = h;
#pragma unroll
                    for (int k = 0; k < A; ++k) acc[k] = __ffma2_rn(w2[k][q], h, acc[k]);
                    if (FVP) {
                        float2 dpre = vb1[q];
#pragma unroll
                        for (int f = 0; f < F; ++f) dpre = __ffma2_rn(vw1[q][f], x[f], dpre);
                        const float2 dh = f2(h.x > 0.0f ? dpre.x : 0.0f, h.y > 0.0f ? dpre.y : 0.0f);
#pragma unroll
                        for (int k = 0; k < A; ++k) accd[k] = __ffma2_rn(vw2[k][q], h, __ffma2_rn(w2[k][q], dh, accd[k]));
                    }
                }
#pragma unroll
                for (int k = 0; k < A; ++k) {
                    pz[k][i] = acc[k].x + acc[k].y;
                    if (FVP) pzd[k][i] = accd[k].x + accd[k].y;
                }
            }
            // ---- reduce across lanes: group g ends up with the logits of sample CH*c + g ----
            float z[A], zd[A];
#pragma unroll
            for (int k = 0; k < A; ++k) {
                z[k] = reduce_scatter<CH>(pz[k], lane) + b2[k];
                zd[k] = FVP ? reduce_scatter<CH>(pzd[k], lane) + vb2[k] : 0.0f;
            }
            // per-sample scalars of that sample live in lane CH*c + g
            const int owner = c * CH + quad_sample;
            const bool s_valid = (valid_mask >> owner) & 1u;
            const int act_s = M::USES_ACT ? __shfl_sync(0xffffffffu, my_act, owner) : 0;
            float adv_s = 0.0f, tgt_s = 0.0f, lp0[2] = {0.0f, 0.0f};
            if (M::USES_ADV) adv_s = __shfl_sync(0xffffffffu, my_adv, owner);
            if (M::USES_LP0) {
                lp0[0] = __shfl_sync(0xffffffffu, my_lp0[0], owner);
                lp0[1] = __shfl_sync(0xffffffffu, my_lp0[1], owner);
            }
            if (M::USES_TARGET) tgt_s = __shfl_sync(0xffffffffu, my_tgt, owner);

            // ---- per-sample algebra (all lanes of a group compute the same values) ----
            float dz[A];
#pragma unroll
            for (int k = 0; k < A; ++k) dz[k] = 0.0f;
            if (s_valid) {
                float lp[A];
                const SampleLoss s = sample_loss<MODE, A>(z, zd, A, act_s, adv_s, tgt_s, make_float2(a.clip_lo, a.clip_hi),
                                                          [&](int k) { return k == 1 ? lp0[1] : lp0[0]; }, lp, dz);
                if (MODE == RL_PASS_STATS && quad_leader)
                    reinterpret_cast<float2 *>(a.logp0)[tile * 32 + owner] = make_float2(lp[0], A > 1 ? lp[A > 1 ? 1 : 0] : 0.0f);
                if (quad_leader) {
                    sc[SC_COUNT] += 1.0;
                    sc[SC_LOSS] += (double)s.loss;
                    sc[SC_KL] += (double)s.kl;
                    sc[SC_ENTROPY] += (double)s.entropy;
#pragma unroll
                    for (int k = 0; k < A; ++k) gb2[k] += (double)dz[k];
                }
            }

            // ---- backward for the same samples ----
            if (BACKWARD) {
#pragma unroll
                for (int i = 0; i < CH; ++i) {
                    float2 d[A];
#pragma unroll
                    for (int k = 0; k < A; ++k) d[k] = dup2(__shfl_sync(0xffffffffu, dz[k], GROUP * i));
                    float2 x[XS / 2];
#pragma unroll
                    for (int v = 0; v < XS / 4; ++v) {
                        const float4 t4 = reinterpret_cast<const float4 *>(xs)[(c * CH + i) * (XS / 4) + v];
                        x[2 * v] = f2(t4.x, t4.y);
                        x[2 * v + 1] = f2(t4.z, t4.w);
                    }
#pragma unroll
                    for (int q = 0; q < NP; ++q) {
                        const float2 h = hid[i][q];
                        float2 dh = __fmul2_rn(d[0], w2[0][q]);
#pragma unroll
                        for (int k = 0; k < A; ++k) {
                            gw2[k][q] = __ffma2_rn(d[k], h, gw2[k][q]);
                            if (k > 0) dh = __ffma2_rn(d[k], w2[k][q], dh);
                        }
                        dh = f2(h.x > 0.0f ? dh.x : 0.0f, h.y > 0.0f ? dh.y : 0.0f);  // relu'(pre)
                        gb1[q] = __fadd2_rn(gb1[q], dh);
#pragma unroll
                        for (int f = 0; f < F; ++f) gw1[q][f] = __ffma2_rn(dh, x[f], gw1[q][f]);
                    }
                }
            }
        }
        if (BACKWARD && ++since_flush == FLUSH_TILES) {
            flush();
            since_flush = 0;
        }
    }
    flush();

    // ---- block reduction into one partial row ----
    double *red = reinterpret_cast<double *>(xs_all);  // reuse the tile region: [nwarps][NSCALAR + A]
    __syncthreads();
#pragma unroll
    for (int k = 0; k < NSCALAR; ++k) {
        const double s = warp_sum_f64(sc[k]);
        if (lane == 0) red[warp * (NSCALAR + A) + k] = s;
    }
#pragma unroll
    for (int k = 0; k < A; ++k) {
        const double s = warp_sum_f64(gb2[k]);
        if (lane == 0) red[warp * (NSCALAR + A) + NSCALAR + k] = s;
    }
    __syncthreads();
    double *row = a.partials + (size_t)blockIdx.x * W;
    for (int i = threadIdx.x; i < W; i += blockDim.x) {
        double s = 0.0;
        if (i < P - A) {
            if (BACKWARD)
                for (int w = 0; w < nwarps; ++w) s += tot_all[(size_t)w * P + i];
        } else if (i < P) {
            if (BACKWARD)
                for (int w = 0; w < nwarps; ++w) s += red[w * (NSCALAR + A) + NSCALAR + (i - (P - A))];
        } else {
            for (int w = 0; w < nwarps; ++w) s += red[w * (NSCALAR + A) + (i - P)];
        }
        row[i] = s;
    }
}

#include "pass_tc.cuh"

// ------------------------------------------------------------------------------------------------
// mlp_pass_any_kernel<MODE>: the same passes for ANY one-hidden-layer module of the reference's MlpConfig
// (mlp.rs:21-61: run-time features F <= 64, hidden units H <= 1024, outputs A <= 16; ReLU / sigmoid / tanh /
// identity), so that TRPO / PPO / REINFORCE / critic / DQN updates also serve Chain, MemoryGame, the bandit
// meta-env and non-default CartPole networks.  Same contract as mlp_pass_kernel (one f64 partial row per CTA),
// different shape of work: sizes are run-time values, so nothing is register-blocked -- a warp owns tiles of 32
// samples and walks them one by one; lane l owns hidden units {l + 32 u}; parameters (W1 transposed to [F][H] so
// that lanes read consecutive words) and the tile's observations sit in shared memory; logits are combined by an
// xor-butterfly (bit-identical in every lane); the backward sweep recomputes a unit's pre-activation instead of
// keeping it, and adds this lane's gradient entries straight into the warp's f64 totals in shared memory (each
// entry has one owner lane: no atomics, fixed order).  Correctness-first fallback: ~5-10x slower per sample than the
// tensor-core passes of the default networks.
// ------------------------------------------------------------------------------------------------
constexpr int ANY_MAXA = 16, ANY_MAXF = 64, ANY_MAXH = 1024, ANY_THREADS = 128;
constexpr size_t ANY_SMEM_CAP = 200 * 1024;
struct AnyShape {
    int F, H, A, act;
    int L;      // hidden layers (MlpConfig::hidden_sizes); H = Hs[0]
    int Hs[3];
};

// Layer-generic (L = 2 or 3) form of the same kernel: every Linear's weights sit in shared memory TRANSPOSED as
// [input][unit] with an odd row pitch, so that both the forward sweep (lanes over units, fixed input) and the backward
// sweep of the layer above (lanes over inputs, fixed unit) are conflict-free; the warp's f64 totals use the same layout;
// activations, tangents and deltas of the sample in flight live in per-warp buffers of ANY_DEEP_MAXH floats.
constexpr int ANY_DEEP_MAXH = 256;
__host__ __device__ inline DeepLayout deep_layout(const AnyShape &sh) { return rl_mlp_layout(sh.F, sh.L, sh.Hs, sh.A); }

// floats per activation / tangent / delta buffer: the widest hidden layer, rounded up to a multiple of 32
__host__ __device__ inline int any_buf_stride(const DeepLayout &d) { return (d.maxH + 31) / 32 * 32; }

__host__ __device__ inline size_t any_smem_bytes(const AnyShape &sh, int nwarps, bool backward, bool fvp) {
    const DeepLayout d = deep_layout(sh);
    const size_t Pp = (size_t)d.P_pad;
    // totals | scalars | theta (+ direction) | tile observations | per warp, for two samples in flight: h[L], tangent[L], delta[2]
    return (backward ? (size_t)nwarps * Pp * sizeof(double) : 0) + (size_t)nwarps * (NSCALAR + ANY_MAXA) * sizeof(double) +
           Pp * sizeof(float) * (fvp ? 2 : 1) + (size_t)nwarps * 32 * sh.F * sizeof(float) +
           (size_t)nwarps * 2 * (2 * sh.L + 2) * any_buf_stride(d) * sizeof(float);
}

__device__ __forceinline__ float warp_allsum_f32(float x) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    return x;
}

// The kernel's inner loops.  One warp per scheduler runs this kernel (its f64 totals fill shared memory), so the loops are
// written for instruction economy and independent work: TWO samples share every weight / total they touch, and each
// result is built from two independent partial sums (same products, additions regrouped).
__device__ __forceinline__ void any_dot2(const float *__restrict__ w, int stride, const float *__restrict__ v0,
                                         const float *__restrict__ v1, int n, float init0, float init1, float &r0, float &r1) {
    float a0 = init0, a1 = 0.0f, b0 = init1, b1 = 0.0f;
    int f = 0;
    for (; f + 1 < n; f += 2) {
        const float w0 = w[f * stride], w1 = w[(f + 1) * stride];
        a0 = fmaf(w0, v0[f], a0); b0 = fmaf(w0, v1[f], b0);
        a1 = fmaf(w1, v0[f + 1], a1); b1 = fmaf(w1, v1[f + 1], b1);
    }
    if (f < n) {
        const float w0 = w[f * stride];
        a0 = fmaf(w0, v0[f], a0); b0 = fmaf(w0, v1[f], b0);
    }
    r0 = a0 + a1;
    r1 = b0 + b1;
}
// tot[f * stride] += d0 * v0[f] + d1 * v1[f]  (f64 totals, each entry owned by this lane)
__device__ __forceinline__ void any_axpy2(double *__restrict__ tot, int stride, float d0, const float *__restrict__ v0, float d1,
                                          const float *__restrict__ v1, int n) {
    int f = 0;
    for (; f + 1 < n; f += 2) {
        double t0 = tot[f * stride], t1 = tot[(f + 1) * stride];
        t0 += (double)fmaf(d1, v1[f], d0 * v0[f]);
        t1 += (double)fmaf(d1, v1[f + 1], d0 * v0[f + 1]);
        tot[f * stride] = t0;
        tot[(f + 1) * stride] = t1;
    }
    if (f < n) tot[f * stride] += (double)fmaf(d1, v1[f], d0 * v0[f]);
}

template <int MODE>
__global__ void __launch_bounds__(ANY_THREADS) mlp_pass_any_kernel(PassArgs a, AnyShape sh) {
    using M = PassMode<MODE>;
    constexpr bool BACKWARD = M::BACKWARD, FVP = M::FVP;
    constexpr int SB = 2;  // samples in flight per warp
    if (a.skip_flag && *a.skip_flag) return;
    const int F = sh.F, A = sh.A, act = sh.act, LL = sh.L;
    const DeepLayout dl = deep_layout(sh);
    const int P = dl.P, W = P + NSCALAR, PL = dl.P_pad, HB = any_buf_stride(dl);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;

    extern __shared__ __align__(16) unsigned char any_smem[];
    double *tot_all = reinterpret_cast<double *>(any_smem);                        // [nwarps][PL], every Linear as [input][unit]
    double *red = tot_all + (BACKWARD ? (size_t)nwarps * PL : 0);                  // [nwarps][NSCALAR + ANY_MAXA]
    float *th = reinterpret_cast<float *>(red + (size_t)nwarps * (NSCALAR + ANY_MAXA));  // theta, same layout
    float *tv = th + PL;                                                           // FVP: the direction, same layout
    float *xs_all = th + (FVP ? 2 : 1) * (size_t)PL;
    float *xs = xs_all + (size_t)warp * 32 * F;
    // per warp and sample in flight: activations h[L], their tangents [L], two delta buffers; HB floats each
    float *bufs = xs_all + (size_t)nwarps * 32 * F + (size_t)warp * SB * (2 * LL + 2) * HB;
    auto buf = [&](int which, int b) { return bufs + ((size_t)b * (2 * LL + 2) + which) * HB; };
    double *tot = tot_all + (size_t)warp * PL;
    for (int i = threadIdx.x; i < P; i += blockDim.x) {
        const int dst = deep_pidx(dl, i);
        th[dst] = a.theta[i];
        if (FVP) tv[dst] = a.vec[i];
    }
    if (BACKWARD)
        for (int i = lane; i < PL; i += 32) tot[i] = 0.0;
    __syncthreads();

    double gb2[ANY_MAXA], sc[NSCALAR];  // lane 0's copies are the ones reported (every lane computes the same values)
#pragma unroll
    for (int k = 0; k < ANY_MAXA; ++k) gb2[k] = 0.0;
#pragma unroll
    for (int k = 0; k < NSCALAR; ++k) sc[k] = 0.0;

    const uint64_t TE = a.T * a.E, ntiles = (TE + 31) / 32;
    const uint64_t warp_global = (uint64_t)blockIdx.x * nwarps + warp, total_warps = (uint64_t)gridDim.x * nwarps;
    for (uint64_t tile = warp_global; tile < ntiles; tile += total_warps) {
        const uint64_t n = tile * 32 + lane;
        const bool in_range = n < TE;
        const uint64_t t = in_range ? n / a.E : 0, e = in_range ? n - t * a.E : 0;
        const bool valid = in_range && a.succ[n] != RL_PAD;
        __syncwarp();
        for (int f = 0; f < F; ++f) xs[lane * F + f] = valid ? __ldg(a.obs + (t * F + f) * a.E + e) : 0.0f;
        const int my_act = (M::USES_ACT && valid) ? (int)a.action[n] : 0;
        const float my_adv = (M::USES_ADV && valid) ? a.adv[n] : 0.0f;
        const float my_tgt = (M::USES_TARGET && valid) ? a.target[n] : 0.0f;
        unsigned todo = __ballot_sync(0xffffffffu, valid);
        __syncwarp();
        while (todo) {  // warp-uniform: the next two valid samples of the tile (the last one may be alone)
            const int s0 = __ffs(todo) - 1;
            todo &= todo - 1;
            const bool two = todo != 0;
            const int s1 = two ? __ffs(todo) - 1 : s0;
            if (two) todo &= todo - 1;
            const int sidx[SB] = {s0, s1};
            const float *x0 = xs + s0 * F, *x1 = xs + s1 * F;
            // ---- forward: lane j owns units {j + 32 u} of every layer; outputs (and tangents) go to the warp's buffers ----
            const float *vin0 = x0, *vin1 = x1, *dvin0 = nullptr, *dvin1 = nullptr;
            for (int l = 0; l < LL; ++l) {
                const int n_in = dl.in[l], n_out = dl.out[l], ld = dl.ld[l];
                const float *Wt = th + dl.off_w[l], *bb = th + dl.off_b[l];
                const float *vWt = tv + dl.off_w[l], *vbb = tv + dl.off_b[l];
                float *h0 = buf(l, 0), *h1 = buf(l, 1), *d0 = buf(LL + l, 0), *d1 = buf(LL + l, 1);
                for (int j = lane; j < n_out; j += 32) {
                    float p0, p1;
                    any_dot2(Wt + j, ld, vin0, vin1, n_in, bb[j], bb[j], p0, p1);
                    const float a0 = rl_activate(act, p0), a1 = rl_activate(act, p1);
                    h0[j] = a0;
                    h1[j] = a1;
                    if (FVP) {
                        float q0, q1;
                        any_dot2(vWt + j, ld, vin0, vin1, n_in, vbb[j], vbb[j], q0, q1);
                        if (dvin0) any_dot2(Wt + j, ld, dvin0, dvin1, n_in, q0, q1, q0, q1);
                        d0[j] = act_grad(act, a0, a0) * q0;
                        d1[j] = act_grad(act, a1, a1) * q1;
                    }
                }
                __syncwarp();
                vin0 = h0; vin1 = h1;
                dvin0 = d0; dvin1 = d1;
            }
            // output Linear: partial sums over this lane's units of the last hidden layer, then a butterfly
            float zz[SB][ANY_MAXA], zzd[SB][FVP ? ANY_MAXA : 1], dzz[SB][ANY_MAXA];
            {
                float pz[SB][ANY_MAXA], pzd[SB][FVP ? ANY_MAXA : 1];
#pragma unroll
                for (int b = 0; b < SB; ++b)
#pragma unroll
                    for (int k = 0; k < ANY_MAXA; ++k) {
                        pz[b][k] = 0.0f;
                        if (FVP) pzd[b][k] = 0.0f;
                    }
                const int n_in = dl.in[LL], ld = dl.ld[LL];
                const float *Wt = th + dl.off_w[LL], *vWt = tv + dl.off_w[LL];
                for (int j = lane; j < n_in; j += 32) {
                    const float hv[SB] = {vin0[j], vin1[j]};
                    const float dv[SB] = {FVP ? dvin0[j] : 0.0f, FVP ? dvin1[j] : 0.0f};
#pragma unroll
                    for (int k = 0; k < ANY_MAXA; ++k)
                        if (k < A) {
                            const float wk = Wt[j * ld + k], vwk = FVP ? vWt[j * ld + k] : 0.0f;
#pragma unroll
                            for (int b = 0; b < SB; ++b) {
                                pz[b][k] = fmaf(wk, hv[b], pz[b][k]);
                                if (FVP) pzd[b][k] = fmaf(vwk, hv[b], fmaf(wk, dv[b], pzd[b][k]));
                            }
                        }
                }
                const float *b_out = th + dl.off_b[LL], *vb_out = tv + dl.off_b[LL];
#pragma unroll
                for (int b = 0; b < SB; ++b)
#pragma unroll
                    for (int k = 0; k < ANY_MAXA; ++k) {
                        zz[b][k] = k < A ? warp_allsum_f32(pz[b][k]) + b_out[k] : 0.0f;
                        if (FVP) zzd[b][k] = k < A ? warp_allsum_f32(pzd[b][k]) + vb_out[k] : 0.0f;
                    }
            }
            // ---- per-sample algebra (every lane computes the same values) ----
#pragma unroll
            for (int b = 0; b < SB; ++b) {
#pragma unroll
                for (int k = 0; k < ANY_MAXA; ++k) dzz[b][k] = 0.0f;
                if (b == 1 && !two) continue;  // (warp-uniform) no second sample: its logit gradients stay zero
                const uint64_t ns = tile * 32 + sidx[b];
                const int act_s = __shfl_sync(0xffffffffu, my_act, sidx[b]);
                const float adv_s = __shfl_sync(0xffffffffu, my_adv, sidx[b]), tgt_s = __shfl_sync(0xffffffffu, my_tgt, sidx[b]);
                // the behaviour log-probabilities in registers, each read once; the taken action's by a search
                float lp[ANY_MAXA], lp0[M::USES_LP0 ? ANY_MAXA : 1];
                if (M::USES_LP0) {
#pragma unroll
                    for (int k = 0; k < ANY_MAXA; ++k) lp0[k] = k < A ? a.logp0[ns * A + k] : 0.0f;
                }
                auto lp0_at = [&](int k) {
                    float v = 0.0f;
#pragma unroll
                    for (int j = 0; j < ANY_MAXA; ++j)
                        if (j == k) v = lp0[j];
                    return v;
                };
                const SampleLoss s = sample_loss<MODE, ANY_MAXA>(zz[b], zzd[b], A, act_s, adv_s, tgt_s, make_float2(a.clip_lo, a.clip_hi),
                                                                 lp0_at, lp, dzz[b]);
                if (MODE == RL_PASS_STATS) {
#pragma unroll
                    for (int k = 0; k < ANY_MAXA; ++k)
                        if (k < A && lane == k) a.logp0[ns * A + k] = lp[k];
                }
                sc[SC_COUNT] += 1.0;
                sc[SC_LOSS] += (double)s.loss;
                sc[SC_KL] += (double)s.kl;
                sc[SC_ENTROPY] += (double)s.entropy;
#pragma unroll
                for (int k = 0; k < ANY_MAXA; ++k) gb2[k] += (double)dzz[b][k];
            }

            // ---- backward: this lane's units, straight into the warp's f64 totals (one update per entry for both samples) ----
            if (BACKWARD) {
                float *delta0 = buf(2 * LL, 0), *delta1 = buf(2 * LL, 1), *next0 = buf(2 * LL + 1, 0), *next1 = buf(2 * LL + 1, 1);
                {   // output Linear: gradients of its weights, delta of the last hidden layer
                    const int n_in = dl.in[LL], ld = dl.ld[LL];
                    const float *Wt = th + dl.off_w[LL];
                    for (int j = lane; j < n_in; j += 32) {
                        const float hv0 = vin0[j], hv1 = vin1[j];
                        float dh0 = 0.0f, dh1 = 0.0f;
#pragma unroll
                        for (int k = 0; k < ANY_MAXA; ++k)
                            if (k < A) {
                                const float wk = Wt[j * ld + k];
                                dh0 = fmaf(dzz[0][k], wk, dh0);
                                dh1 = fmaf(dzz[1][k], wk, dh1);
                                tot[dl.off_w[LL] + j * ld + k] += (double)fmaf(dzz[1][k], hv1, dzz[0][k] * hv0);
                            }
                        delta0[j] = dh0 * act_grad(act, hv0, hv0);
                        delta1[j] = dh1 * act_grad(act, hv1, hv1);
                    }
                    __syncwarp();
                }
                for (int l = LL - 1; l >= 0; --l) {
                    const int n_in = dl.in[l], n_out = dl.out[l], ld = dl.ld[l];
                    const float *in0 = l == 0 ? x0 : buf(l - 1, 0), *in1 = l == 0 ? x1 : buf(l - 1, 1);
                    for (int j = lane; j < n_out; j += 32) {
                        const float dj0 = delta0[j], dj1 = delta1[j];
                        tot[dl.off_b[l] + j] += (double)(dj0 + dj1);
                        any_axpy2(tot + dl.off_w[l] + j, ld, dj0, in0, dj1, in1, n_in);
                    }
                    if (l > 0) {  // delta of the layer below: lane i owns ITS unit i (= input i of this layer)
                        const float *Wt = th + dl.off_w[l];
                        for (int i2 = lane; i2 < n_in; i2 += 32) {
                            float acc0, acc1;
                            any_dot2(Wt + i2 * ld, 1, delta0, delta1, n_out, 0.0f, 0.0f, acc0, acc1);
                            next0[i2] = acc0 * act_grad(act, in0[i2], in0[i2]);
                            next1[i2] = acc1 * act_grad(act, in1[i2], in1[i2]);
                        }
                        __syncwarp();
                        float *t0 = delta0; delta0 = next0; next0 = t0;
                        float *t1 = delta1; delta1 = next1; next1 = t1;
                    }
                }
                __syncwarp();
            }
        }
    }

    // ---- block reduction into one partial row (parameter order of Module::variables) ----
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < NSCALAR; ++k) red[warp * (NSCALAR + ANY_MAXA) + k] = sc[k];
#pragma unroll
        for (int k = 0; k < ANY_MAXA; ++k) red[warp * (NSCALAR + ANY_MAXA) + NSCALAR + k] = gb2[k];
    }
    __syncthreads();
    double *row = a.partials + (size_t)blockIdx.x * W;
    for (int i = threadIdx.x; i < W; i += blockDim.x) {
        double s = 0.0;
        if (i < P - A) {
            const int src = deep_pidx(dl, i);
            if (BACKWARD)
                for (int w = 0; w < nwarps; ++w) s += tot_all[(size_t)w * PL + src];
        } else if (i < P) {
            if (BACKWARD)
                for (int w = 0; w < nwarps; ++w) s += red[w * (NSCALAR + ANY_MAXA) + NSCALAR + (i - (P - A))];
        } else {
            for (int w = 0; w < nwarps; ++w) s += red[w * (NSCALAR + ANY_MAXA) + (i - P)];
        }
        row[i] = s;
    }
}


// rows[B][W] -> out[W] in a fixed summation order.  A block owns 32 columns; warp w sums rows
// w, w + 8, ... (independent coalesced 256 B loads), then the 8 partials are added in warp order.
__global__ void __launch_bounds__(256) reduce_rows_kernel(const double *__restrict__ rows, int B, int W,
                                                         double *__restrict__ out, const int *skip_flag) {
    if (skip_flag && *skip_flag) return;
    __shared__ double part[8][32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int col = blockIdx.x * 32 + lane;
    double s = 0.0;
    if (col < W) {
#pragma unroll 8
        for (int b = warp; b < B; b += 8) s += rows[(size_t)b * W + col];
    }
    part[warp][lane] = s;
    __syncthreads();
    if (warp == 0 && col < W) {
        double t = 0.0;
#pragma unroll
        for (int w = 0; w < 8; ++w) t += part[w][lane];
        out[col] = t;
    }
}

// ------------------------------------------------------------------------------------------------
// single-CTA vector kernels
// ------------------------------------------------------------------------------------------------
struct TrpoState {
    double N, loss0, entropy, rr, step_size, step_scale, loss_final, kl_final;
    int cg_done, cg_iters, accepted, num_backtracks, status, evals;
};

constexpr int VEC_THREADS = 1024;

__device__ double block_sum_f64(double v) {
    __shared__ double red[32];
    __shared__ double result;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v = warp_sum_f64(v);
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    if (warp == 0) {
        double s = lane < (int)(blockDim.x >> 5) ? red[lane] : 0.0;
        s = warp_sum_f64(s);
        if (lane == 0) result = s;
    }
    __syncthreads();
    return result;
}

__global__ void trpo_begin_kernel(TrpoState *st, const double *sums, int P) {
    if (threadIdx.x == 0) {
        st->N = sums[P + SC_COUNT];
        st->entropy = sums[P + SC_ENTROPY] / st->N;
        st->cg_done = 0; st->cg_iters = 0; st->accepted = 0; st->num_backtracks = -1; st->status = RL_OK; st->evals = 0;
        st->step_size = 0.0; st->step_scale = 0.0; st->rr = 0.0;
        st->loss0 = 0.0; st->loss_final = 0.0; st->kl_final = INFINITY;
    }
}

// g = grad / N; x = 0; r = p = g; rr = r.r  (conjugate_gradient.rs:121-143,377-384)
__global__ void __launch_bounds__(VEC_THREADS)
    trpo_cg_init_kernel(TrpoState *st, const double *sums, int P, float *g, float *x, float *r, float *p,
                        const float *theta, float *theta0) {
    const double N = st->N;
    double acc = 0.0;
    for (int i = threadIdx.x; i < P; i += blockDim.x) {
        const float gi = (float)(sums[i] / N);
        g[i] = gi; x[i] = 0.0f; r[i] = gi; p[i] = gi;
        theta0[i] = theta[i];
        acc += (double)gi * (double)gi;
    }
    const double rr = block_sum_f64(acc);
    if (threadIdx.x == 0) {
        st->rr = (double)(float)rr;
        st->loss0 = (double)(float)(sums[P + SC_LOSS] / N);
        st->loss_final = st->loss0;
    }
}

// one CG iteration given the Fisher-vector product of p (conjugate_gradient.rs:386-401, :335-337)
__global__ void __launch_bounds__(VEC_THREADS)
    trpo_cg_step_kernel(TrpoState *st, const double *sums, int P, float *x, float *r, float *p, float reg, double tol) {
    if (st->cg_done) return;
    __shared__ float s_alpha, s_mu;
    __shared__ int s_done;
    const double N = st->N;
    double acc = 0.0;
    for (int i = threadIdx.x; i < P; i += blockDim.x) {
        const float z = __fadd_rn((float)(sums[i] / N), __fmul_rn(p[i], reg));
        acc += (double)p[i] * (double)z;
    }
    const double pz = block_sum_f64(acc);
    if (threadIdx.x == 0) s_alpha = (float)st->rr / (float)pz;
    __syncthreads();
    const float alpha = s_alpha;
    acc = 0.0;
    for (int i = threadIdx.x; i < P; i += blockDim.x) {
        const float z = __fadd_rn((float)(sums[i] / N), __fmul_rn(p[i], reg));
        x[i] = __fadd_rn(x[i], __fmul_rn(alpha, p[i]));
        const float ri = __fadd_rn(r[i], __fmul_rn(-alpha, z));
        r[i] = ri;
        acc += (double)ri * (double)ri;
    }
    const double rr_new = block_sum_f64(acc);
    if (threadIdx.x == 0) {
        const float rrn = (float)rr_new;
        st->cg_iters += 1;
        if ((double)rrn < tol) {
            s_done = 1;
            st->cg_done = 1;
        } else {
            s_done = 0;
            s_mu = rrn / (float)st->rr;
            st->rr = (double)rrn;
        }
    }
    __syncthreads();
    if (!s_done) {
        const float mu = s_mu;
        for (int i = threadIdx.x; i < P; i += blockDim.x) p[i] = __fadd_rn(__fmul_rn(p[i], mu), r[i]);
    }
}

// nan_to_num_(0.0, None, None) on the step direction (conjugate_gradient.rs:152); also re-arms the FVP pass
__global__ void trpo_nan_to_num_kernel(TrpoState *st, float *x, int P) {
    for (int i = threadIdx.x; i < P; i += blockDim.x) {
        float v = x[i];
        if (isnan(v)) v = 0.0f;
        else if (isinf(v)) v = v > 0.0f ? 3.402823466e+38f : -3.402823466e+38f;
        x[i] = v;
    }
    if (threadIdx.x == 0) st->cg_done = 0;  // the step-size FVP must always run
}

// step_size = sqrt(2 delta / (x.Hx + 1e-8)), NaN -> 1; descent = step_size * x  (conjugate_gradient.rs:155-166)
__global__ void __launch_bounds__(VEC_THREADS)
    trpo_step_size_kernel(TrpoState *st, const double *sums, int P, const float *x, float *descent, float reg,
                          double max_kl) {
    __shared__ float s_step;
    const double N = st->N;
    double acc = 0.0;
    for (int i = threadIdx.x; i < P; i += blockDim.x) {
        const float hx = __fadd_rn((float)(sums[i] / N), __fmul_rn(x[i], reg));
        acc += (double)x[i] * (double)hx;
    }
    const double xhx = block_sum_f64(acc);
    if (threadIdx.x == 0) {
        double step = sqrt(1.0 / ((double)(float)xhx + 1e-8) * max_kl * 2.0);
        if (isnan(step)) step = 1.0;
        st->step_size = step;
        s_step = (float)step;
    }
    __syncthreads();
    const float step = s_step;
    for (int i = threadIdx.x; i < P; i += blockDim.x) descent[i] = __fmul_rn(step, x[i]);
}

// theta = theta0 - ratio * descent  (conjugate_gradient.rs:201-213)
__global__ void trpo_ls_candidate_kernel(const TrpoState *st, float *theta, const float *theta0, const float *descent,
                                         float ratio, int P) {
    if (st->accepted) return;
    for (int i = threadIdx.x; i < P; i += blockDim.x) theta[i] = __fsub_rn(theta0[i], __fmul_rn(ratio, descent[i]));
}

// accept iff loss < loss0 && kl <= max_kl  (conjugate_gradient.rs:215-223)
__global__ void trpo_ls_check_kernel(TrpoState *st, const double *sums, int P, double max_kl, int i, double ratio) {
    if (threadIdx.x != 0 || st->accepted) return;
    const double loss = (double)(float)(sums[P + SC_LOSS] / st->N);
    const double kl = (double)(float)(sums[P + SC_KL] / st->N);
    st->loss_final = loss;
    st->kl_final = kl;
    st->evals += 1;
    if (loss < st->loss0 && kl <= max_kl) {
        st->accepted = 1;
        st->num_backtracks = i;
        st->step_scale = ratio;
    }
}

// error classification and parameter rollback (conjugate_gradient.rs:228-251)
__global__ void trpo_ls_finish_kernel(TrpoState *st, float *theta, const float *theta0, int P, double max_kl,
                                      int accept_violation) {
    __shared__ int s_status;
    if (threadIdx.x == 0) {
        const double loss = st->loss_final, kl = st->kl_final;
        int status = RL_OK;
        if (isnan(loss)) status = RL_STEP_NAN_LOSS;
        else if (isnan(kl)) status = RL_STEP_NAN_CONSTRAINT;
        else if (loss >= st->loss0) status = RL_STEP_LOSS_NOT_IMPROVING;
        else if (kl >= max_kl && !accept_violation) status = RL_STEP_CONSTRAINT_VIOLATED;
        st->status = status;
        s_status = status;
    }
    __syncthreads();
    if (s_status != RL_OK)
        for (int i = threadIdx.x; i < P; i += blockDim.x) theta[i] = theta0[i];
}

// libtorch Adam::step (non-amsgrad) on the mean gradient; records the loss of this step
struct AdamArgs {
    double lr, beta1, beta2, weight_decay, eps;
};
__global__ void __launch_bounds__(VEC_THREADS)
    adam_step_kernel(const double *sums, int P, float *theta, float *m, float *v, AdamArgs c, uint64_t step,
                     double *loss_out) {
    const double N = sums[P + SC_COUNT];
    const float beta1 = (float)c.beta1, beta2 = (float)c.beta2;
    const float omb1 = (float)(1.0 - c.beta1), omb2 = (float)(1.0 - c.beta2);
    const double bc1 = 1.0 - pow(c.beta1, (double)step), bc2 = 1.0 - pow(c.beta2, (double)step);
    const float step_size = (float)(c.lr / bc1), bc2_sqrt = (float)sqrt(bc2), eps = (float)c.eps;
    for (int i = threadIdx.x; i < P; i += blockDim.x) {
        float g = (float)(sums[i] / N);
        float th = theta[i];
        if (c.weight_decay != 0.0) g = __fadd_rn(g, __fmul_rn((float)c.weight_decay, th));
        // exp_avg.mul_(beta1).add_(grad, 1 - beta1); exp_avg_sq.mul_(beta2).addcmul_(grad, grad, 1 - beta2)
        const float mi = __fadd_rn(__fmul_rn(m[i], beta1), __fmul_rn(omb1, g));
        const float vi = __fadd_rn(__fmul_rn(v[i], beta2), __fmul_rn(__fmul_rn(omb2, g), g));
        m[i] = mi;
        v[i] = vi;
        const float denom = __fadd_rn(__fdiv_rn(__fsqrt_rn(vi), bc2_sqrt), eps);
        theta[i] = __fadd_rn(th, __fmul_rn(-step_size, __fdiv_rn(mi, denom)));
    }
    if (threadIdx.x == 0 && loss_out) *loss_out = sums[P + SC_LOSS] / N;
}


// reduce_rows_kernel + adam_step_kernel in one launch (single-GPU loops: no all-reduce sits between them).
// Every block reduces its 32 columns exactly as reduce_rows_kernel does, plus the sample-count column, and
// applies libtorch's Adam::step to its own parameters; block 0 also publishes the loss.
__global__ void __launch_bounds__(256)
    reduce_rows_adam_kernel(const double *__restrict__ rows, int B, int W, int P, double *__restrict__ sums, float *theta,
                            float *m, float *v, AdamArgs c, uint64_t step, double *loss_out) {
    __shared__ double part[8][32];
    __shared__ double cnt_part[8], loss_part[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int col = blockIdx.x * 32 + lane;
    double s = 0.0;
    if (col < W) {
#pragma unroll 8
        for (int b = warp; b < B; b += 8) s += rows[(size_t)b * W + col];
    }
    part[warp][lane] = s;
    // the scalar columns every block needs (sample count; loss for block 0): rows spread over all 256 threads.
    // The count is an integer, exact in any order; the loss order is fixed by this loop.
    double cn = 0.0, ls = 0.0;
    for (int b = threadIdx.x; b < B; b += 256) {
        cn += rows[(size_t)b * W + P + SC_COUNT];
        ls += rows[(size_t)b * W + P + SC_LOSS];
    }
    cn = warp_sum_f64(cn);
    ls = warp_sum_f64(ls);
    if (lane == 0) {
        cnt_part[warp] = cn;
        loss_part[warp] = ls;
    }
    __syncthreads();
    if (warp == 0) {
        double t = 0.0, N = 0.0, lsum = 0.0;
#pragma unroll
        for (int w = 0; w < 8; ++w) {
            t += part[w][lane];
            N += cnt_part[w];
            lsum += loss_part[w];
        }
        if (col < W) sums[col] = t;
        if (col < P) {
            const float beta1 = (float)c.beta1, beta2 = (float)c.beta2;
            const float omb1 = (float)(1.0 - c.beta1), omb2 = (float)(1.0 - c.beta2);
            const double bc1 = 1.0 - pow(c.beta1, (double)step), bc2 = 1.0 - pow(c.beta2, (double)step);
            const float step_size = (float)(c.lr / bc1), bc2_sqrt = (float)sqrt(bc2), eps = (float)c.eps;
            float g = (float)(t / N);
            const float th = theta[col];
            if (c.weight_decay != 0.0) g = __fadd_rn(g, __fmul_rn((float)c.weight_decay, th));
            const float mi = __fadd_rn(__fmul_rn(m[col], beta1), __fmul_rn(omb1, g));
            const float vi = __fadd_rn(__fmul_rn(v[col], beta2), __fmul_rn(__fmul_rn(omb2, g), g));
            m[col] = mi;
            v[col] = vi;
            const float denom = __fadd_rn(__fdiv_rn(__fsqrt_rn(vi), bc2_sqrt), eps);
            theta[col] = __fadd_rn(th, __fmul_rn(-step_size, __fdiv_rn(mi, denom)));
        }
        if (blockIdx.x == 0 && lane == 0 && loss_out) *loss_out = lsum / N;
    }
}

// Row reduction fused with the cross-GPU sum (and, for the optimizer loops, with Adam): the multi-GPU form of
// reduce_rows_kernel / reduce_rows_adam_kernel.  Block b reduces its 32 columns over this rank's partial rows, PUSHES
// the 32 sums (+ this rank's sample count and loss) into slot [parity][rank][b] of every peer's mailbox over NVLink,
// publishes the collective's sequence number in the matching flag, then waits on its OWN mailbox for the same slot
// of every source rank and adds the slots in rank order -- the same order on every rank, so all ranks hold
// bit-identical sums and no broadcast is needed.  One launch replaces reduce + ncclAllReduce (+ Adam); the data
// path is 7 KB of peer stores per rank and the waits are local polls.
//   Slot reuse: collective k uses parity k & 1.  A rank can reach collective k + 2 only after it completed k + 1,
// i.e. after every peer posted k + 1, which a peer does (stream order) after it finished reading k.  Skipped passes
// (device-side skip flag, identical on every rank) still run the exchange so that parities stay aligned.
struct XAdam {
    float *theta, *m, *v;
    AdamArgs c;
    uint64_t step;
    double *loss_out;
    int P;
};
template <bool ADAM>
__global__ void __launch_bounds__(256)
    reduce_rows_x_kernel(const double *__restrict__ rows, int B, int W, int P, double *__restrict__ sums, rl_xpeer x,
                         unsigned long long seq, const int *skip_flag, XAdam ad) {
    __shared__ double part[8][32];
    __shared__ double cnt_part[8], loss_part[8];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int col = blockIdx.x * 32 + lane;
    // (a timeout in an earlier reduction is sticky: nothing is written from then on, x_error_check reports it)
    const bool skip = (skip_flag && *skip_flag) || *reinterpret_cast<const volatile int *>(x.error) != 0;
    double s = 0.0;
    if (col < W && !skip) {
#pragma unroll 8
        for (int b = warp; b < B; b += 8) s += rows[(size_t)b * W + col];
    }
    part[warp][lane] = s;
    double cn = 0.0, ls = 0.0;
    if (ADAM && !skip) {
        for (int b = threadIdx.x; b < B; b += 256) {
            cn += rows[(size_t)b * W + P + SC_COUNT];
            ls += rows[(size_t)b * W + P + SC_LOSS];
        }
        cn = warp_sum_f64(cn);
        ls = warp_sum_f64(ls);
    }
    if (lane == 0) {
        cnt_part[warp] = cn;
        loss_part[warp] = ls;
    }
    __syncthreads();
    if (warp != 0) return;
    double t = 0.0, N = 0.0, lsum = 0.0;
#pragma unroll
    for (int w = 0; w < 8; ++w) {
        t += part[w][lane];
        N += cnt_part[w];
        lsum += loss_part[w];
    }
    // ---- push this block's message to every rank (own mailbox included) ----
    const size_t par = (size_t)(seq & 1ull);
    const size_t slot_out = (par * x.world + x.rank) * RL_X_BLOCKS + blockIdx.x;
    for (int p = 0; p < x.world; ++p) {
        double *dst = x.data[p] + slot_out * RL_X_SLOT;
        dst[lane] = t;
        if (lane == 0) {
            dst[32] = N;
            dst[33] = lsum;
        }
    }
    __threadfence_system();
    __syncwarp();
    if (lane < x.world) {
        volatile unsigned long long *f = x.flag[lane] + slot_out;
        *f = seq;
    }
    // ---- wait for every source rank's message in the own mailbox ----
    bool timed_out = false;
    if (lane < x.world) {
        const volatile unsigned long long *f = x.flag[x.rank] + (par * x.world + lane) * RL_X_BLOCKS + blockIdx.x;
        const long long t0 = clock64();
        while (*f != seq) {
            if (clock64() - t0 > 20000000000ll) {  // ~10 s: a peer never arrived
                atomicExch(x.error, 1);
                timed_out = true;
                break;
            }
        }
    }
    // a mailbox that never filled holds stale data: write neither the sums nor the Adam step
    if (__any_sync(0xffffffffu, timed_out)) return;
    __threadfence_system();
    double tot = 0.0, Ntot = 0.0, ltot = 0.0;
    for (int src = 0; src < x.world; ++src) {
        const volatile double *msg = x.data[x.rank] + ((par * x.world + src) * RL_X_BLOCKS + blockIdx.x) * RL_X_SLOT;
        tot += msg[lane];
        Ntot += msg[32];
        ltot += msg[33];
    }
    if (skip) return;
    if (col < W) sums[col] = tot;
    if (ADAM) {
        if (col < ad.P) {
            const AdamArgs &c = ad.c;
            const float beta1 = (float)c.beta1, beta2 = (float)c.beta2;
            const float omb1 = (float)(1.0 - c.beta1), omb2 = (float)(1.0 - c.beta2);
            const double bc1 = 1.0 - pow(c.beta1, (double)ad.step), bc2 = 1.0 - pow(c.beta2, (double)ad.step);
            const float step_size = (float)(c.lr / bc1), bc2_sqrt = (float)sqrt(bc2), eps = (float)c.eps;
            float g = (float)(tot / Ntot);
            const float th = ad.theta[col];
            if (c.weight_decay != 0.0) g = __fadd_rn(g, __fmul_rn((float)c.weight_decay, th));
            const float mi = __fadd_rn(__fmul_rn(ad.m[col], beta1), __fmul_rn(omb1, g));
            const float vi = __fadd_rn(__fmul_rn(ad.v[col], beta2), __fmul_rn(__fmul_rn(omb2, g), g));
            ad.m[col] = mi;
            ad.v[col] = vi;
            const float denom = __fadd_rn(__fdiv_rn(__fsqrt_rn(vi), bc2_sqrt), eps);
            ad.theta[col] = __fadd_rn(th, __fmul_rn(-step_size, __fdiv_rn(mi, denom)));
        }
        if (blockIdx.x == 0 && lane == 0 && ad.loss_out) *ad.loss_out = ltot / Ntot;
    }
}

// ------------------------------------------------------------------------------------------------
// host orchestration
// ------------------------------------------------------------------------------------------------
struct PassPlan {
    int P, W, grid;
    int grid_tc;  // CTAs of the tcgen05 passes (mlp_pass_tc_kernel); the partial rows hold max(grid, grid_tc)
    size_t smem;
    double *partials, *sums;
};

template <int F, int A, int UPL>
size_t pass_smem_bytes() {
    constexpr int H = 32 * UPL, P = H * F + H + A * H + A;
    const int nwarps = PASS_THREADS / 32;
    return (size_t)nwarps * P * sizeof(double) + (size_t)nwarps * 32 * 12 * sizeof(float);
}

// Data-parallel group: did a peer-mailbox wait time out (reduce_rows_x_kernel)?  From the failing reduction on every
// launch of that kernel leaves sums and parameters untouched; the update entry points end with this check and report it.
rl_status x_error_check(rl_ctx *ctx, const char *what) {
    if (ctx->world <= 1 || !ctx->x_ok) return RL_OK;
    int *host;
    RL_TRY(rl_ctx_pinned(ctx, 64, (void **)&host));
    RL_CUDA(ctx, cudaMemcpyAsync(host, ctx->x.error, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (*host)
        return rl_fail(ctx, RL_ERR_NCCL, "%s: a rank of the data-parallel group never arrived at a reduction (peer mailbox wait timed out); "
                       "sums and parameters were left untouched from that reduction on", what);
    return RL_OK;
}

// rows of plan.partials -> plan.sums, summed over the data-parallel group: one fused kernel over the peer
// mailboxes when they are mapped (common.cuh rl_xpeer), else reduce_rows_kernel + ncclAllReduce.
rl_status reduce_over_group(rl_ctx *ctx, const PassPlan &plan, int rows, const int *skip_flag) {
    if (ctx->world > 1 && ctx->x_ok && rl_div_up(plan.W, 32) <= RL_X_BLOCKS) {
        ctx->x_seq += 1;
        RL_LAUNCH(ctx, reduce_rows_x_kernel<false>, rl_div_up(plan.W, 32), 256, 0, plan.partials, rows, plan.W, plan.P, plan.sums,
                  ctx->x, ctx->x_seq, skip_flag, XAdam{});
        return RL_OK;
    }
    RL_LAUNCH(ctx, reduce_rows_kernel, rl_div_up(plan.W, 32), 256, 0, plan.partials, rows, plan.W, plan.sums, skip_flag);
    if (ctx->world > 1) RL_TRY(rl_allreduce_f64_inplace(ctx, plan.sums, (size_t)plan.W));
    return RL_OK;
}

// The default networks' passes on the FP32 pipe (mlp_pass_kernel): the cross-check of the tensor-core kernel, selected by
// RL_PASS_KERNEL=ffma or rl_pass_kernel_select(RL_PASS_KERNEL_FFMA).  Tile-chunk size and CTAs per SM per mode:
// forward-only passes fit 2 CTAs/SM at CH = 8; the critic and Q-loss passes run at CH = 4 with 2 CTAs/SM; the
// gradient / Fisher-vector passes need the registers of 1 CTA/SM.
template <int A, int MODE>
rl_status launch_pass_ffma(rl_ctx *ctx, const PassPlan &plan, PassArgs args, bool reduce) {
    constexpr int F = 5, UPL = 4;
    constexpr bool MSE = MODE == RL_PASS_VALUE || MODE == RL_PASS_QLOSS, FWD = MODE == RL_PASS_STATS || MODE == RL_PASS_EVAL;
    constexpr int CH = MSE ? 4 : 8, MINB = MSE || FWD ? 2 : 1;
    const size_t smem = pass_smem_bytes<F, A, UPL>();
    static bool configured = false;
    if (!configured) {
        RL_CUDA(ctx, cudaFuncSetAttribute(mlp_pass_kernel<F, A, UPL, MODE, CH, MINB>,
                                          cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured = true;
    }
    args.partials = plan.partials;
    RL_LAUNCH(ctx, (mlp_pass_kernel<F, A, UPL, MODE, CH, MINB>), plan.grid, PASS_THREADS, smem, args);
    if (!reduce) return RL_OK;
    return reduce_over_group(ctx, plan, plan.grid, args.skip_flag);
}

// Which kernel runs the default networks' passes (RL_PASS_KERNEL_*): RL_PASS_KERNEL from the environment until
// rl_pass_kernel_select sets it.  pass_net_for reads it into the PassNet of an update.
int g_pass_kernel = -1;
int pass_kernel() {
    if (g_pass_kernel < 0) {
        const char *e = getenv("RL_PASS_KERNEL");
        g_pass_kernel = (e && (e[0] == 'f' || e[0] == '0')) ? RL_PASS_KERNEL_FFMA : RL_PASS_KERNEL_TCGEN05;
    }
    return g_pass_kernel;
}
// CTAs of a tensor-core pass: the plan's count (3 per SM) capped at what the mode keeps resident per SM
template <int A, int MODE>
int tc_grid(const rl_ctx *ctx, const PassPlan &plan) {
    const int cap = ctx->sm_count * TcPass<A, MODE>::CTAS_PER_SM;
    return plan.grid_tc < cap ? plan.grid_tc : cap;
}

template <int A, int MODE>
rl_status launch_pass_tc(rl_ctx *ctx, const PassPlan &plan, PassArgs args, bool reduce) {
    constexpr int smem = TcPass<A, MODE>::SMEM;
    static bool configured = false;
    if (!configured) {
        RL_CUDA(ctx, cudaFuncSetAttribute(mlp_pass_tc_kernel<A, MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        configured = true;
    }
    args.partials = plan.partials;
    const int grid = tc_grid<A, MODE>(ctx, plan);
    RL_LAUNCH(ctx, (mlp_pass_tc_kernel<A, MODE>), grid, tc::TC_THREADS, smem, args);
    if (!reduce) return RL_OK;
    return reduce_over_group(ctx, plan, grid, args.skip_flag);
}

rl_status make_plan(rl_ctx *ctx, int P, uint64_t TE, PassPlan *plan, size_t extra_bytes, void **extra) {
    plan->P = P;
    plan->W = P + NSCALAR;
    const uint64_t ntiles = (TE + 31) / 32;
    const uint64_t want = (ntiles + (PASS_THREADS / 32) - 1) / (PASS_THREADS / 32);
    const uint64_t cap = (uint64_t)ctx->sm_count * 2;  // persistent: 2 CTAs per SM (the FVP pass fits 1 and runs 2 waves)
    plan->grid = (int)(want < cap ? (want ? want : 1) : cap);
    const uint64_t tiles_tc = (TE + tc::TC_THREADS - 1) / tc::TC_THREADS, cap_tc = (uint64_t)ctx->sm_count * tc::TC_CTAS_PER_SM;
    plan->grid_tc = (int)(tiles_tc < cap_tc ? (tiles_tc ? tiles_tc : 1) : cap_tc);
    const size_t rows = (size_t)(plan->grid > plan->grid_tc ? plan->grid : plan->grid_tc) * plan->W * sizeof(double),
                 sums = (size_t)plan->W * sizeof(double);
    char *buf;
    RL_TRY(rl_ctx_scratch(ctx, rows + sums + extra_bytes + 256, (void **)&buf));
    plan->partials = (double *)buf;
    plan->sums = (double *)(buf + rows);
    if (extra) *extra = buf + rows + ((sums + 255) / 256) * 256;
    return RL_OK;
}

// ------------------------------------------------------------------------------------------------
// Run-time dispatch over module shapes: the reference's default networks (5 -> 128 -> 1 critic, 5 -> 128 -> 2 policy /
// action-value network, ReLU) take the kernels above (tensor cores, or the FP32 pipe when selected); every other
// module takes mlp_pass_any_kernel.
// ------------------------------------------------------------------------------------------------
struct PassNet {
    bool deflt;
    AnyShape sh;
    int kernel;  // RL_PASS_KERNEL_* of a default network
};

rl_status pass_net_for(rl_ctx *ctx, const rl_mlp *m, int F_data, const char *what, PassNet *out) {
    if (m->in_dim != F_data)
        return rl_fail(ctx, RL_ERR_INVALID_ARG, "%s: a %d->%d->%d module does not match observations of %d features", what,
                       m->in_dim, m->hidden, m->out_dim, F_data);
    out->sh = AnyShape{m->in_dim, m->hidden, m->out_dim, (int)m->act, m->n_hidden, {m->hid[0], m->hid[1], m->hid[2]}};
    out->deflt = m->n_hidden == 1 && F_data == 5 && m->hidden == 128 && m->act == RL_ACT_RELU && (m->out_dim == 1 || m->out_dim == 2);
    out->kernel = pass_kernel();
    if (m->n_hidden > 1) {
        bool ok = m->in_dim >= 1 && m->in_dim <= ANY_MAXF && m->out_dim >= 1 && m->out_dim <= ANY_MAXA;
        for (int l = 0; l < m->n_hidden; ++l) ok = ok && m->hid[l] >= 1 && m->hid[l] <= ANY_DEEP_MAXH;
        if (!ok || any_smem_bytes(out->sh, 1, true, true) > ANY_SMEM_CAP)
            return rl_fail(ctx, RL_ERR_UNSUPPORTED,
                           "%s: modules with two or three hidden layers are built for <= %d features, <= %d units per layer, <= %d "
                           "outputs and <= ~12 K parameters", what, ANY_MAXF, ANY_DEEP_MAXH, ANY_MAXA);
        return RL_OK;
    }
    if (!out->deflt && !(m->in_dim >= 1 && m->in_dim <= ANY_MAXF && m->hidden >= 1 && m->hidden <= ANY_MAXH && m->out_dim >= 1 &&
                         m->out_dim <= ANY_MAXA && any_smem_bytes(out->sh, 1, true, true) <= ANY_SMEM_CAP))
        return rl_fail(ctx, RL_ERR_UNSUPPORTED,
                       "%s: built for one-hidden-layer modules with <= %d features, <= %d units, <= %d outputs and "
                       "<= ~12 K parameters (got %d->%d->%d)", what, ANY_MAXF, ANY_MAXH, ANY_MAXA, m->in_dim, m->hidden, m->out_dim);
    return RL_OK;
}

template <int MODE>
rl_status launch_pass_any_mode(rl_ctx *ctx, const PassPlan &plan, PassArgs args, const AnyShape &sh, bool reduce) {
    int nwarps = ANY_THREADS / 32;
    while (nwarps > 1 && any_smem_bytes(sh, nwarps, pass_backward(MODE), MODE == RL_PASS_FVP) > ANY_SMEM_CAP) nwarps >>= 1;
    const size_t smem = any_smem_bytes(sh, nwarps, pass_backward(MODE), MODE == RL_PASS_FVP);
    static bool configured = false;
    if (!configured) {
        RL_CUDA(ctx, cudaFuncSetAttribute(mlp_pass_any_kernel<MODE>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)ANY_SMEM_CAP));
        configured = true;
    }
    args.partials = plan.partials;
    RL_LAUNCH(ctx, (mlp_pass_any_kernel<MODE>), plan.grid, nwarps * 32, smem, args, sh);
    if (!reduce) return RL_OK;
    return reduce_over_group(ctx, plan, plan.grid, args.skip_flag);
}

// One full-batch pass of `pn` in MODE; *rows = partial rows it wrote.  The critic pass of the default 5 -> 128 -> 1
// network and every other pass of the default 5 -> 128 -> 2 network run on the tensor cores, or on the FP32 pipe when
// pn.kernel selects it; every other module runs on mlp_pass_any_kernel.
template <int MODE>
rl_status launch_pass(rl_ctx *ctx, const PassPlan &plan, const PassArgs &pa, const PassNet &pn, bool reduce, int *rows) {
    constexpr int A = MODE == RL_PASS_VALUE ? 1 : 2;
    if (pn.deflt && pn.sh.A == A && pn.kernel == RL_PASS_KERNEL_TCGEN05) {
        if (rows) *rows = tc_grid<A, MODE>(ctx, plan);
        return launch_pass_tc<A, MODE>(ctx, plan, pa, reduce);
    }
    if (rows) *rows = plan.grid;
    if (pn.deflt && pn.sh.A == A) return launch_pass_ffma<A, MODE>(ctx, plan, pa, reduce);
    return launch_pass_any_mode<MODE>(ctx, plan, pa, pn.sh, reduce);
}

rl_status launch_pass_rt(rl_ctx *ctx, const PassPlan &plan, const PassArgs &pa, int mode, const PassNet &pn, bool reduce = true,
                         int *rows = nullptr) {
    switch (mode) {
    case RL_PASS_STATS: return launch_pass<RL_PASS_STATS>(ctx, plan, pa, pn, reduce, rows);
    case RL_PASS_EVAL: return launch_pass<RL_PASS_EVAL>(ctx, plan, pa, pn, reduce, rows);
    case RL_PASS_GRAD: return launch_pass<RL_PASS_GRAD>(ctx, plan, pa, pn, reduce, rows);
    case RL_PASS_FVP: return launch_pass<RL_PASS_FVP>(ctx, plan, pa, pn, reduce, rows);
    case RL_PASS_PPO: return launch_pass<RL_PASS_PPO>(ctx, plan, pa, pn, reduce, rows);
    case RL_PASS_REINFORCE: return launch_pass<RL_PASS_REINFORCE>(ctx, plan, pa, pn, reduce, rows);
    case RL_PASS_QLOSS: return launch_pass<RL_PASS_QLOSS>(ctx, plan, pa, pn, reduce, rows);
    case RL_PASS_VALUE: return launch_pass<RL_PASS_VALUE>(ctx, plan, pa, pn, reduce, rows);
    default: return rl_fail(ctx, RL_ERR_INVALID_ARG, "unknown pass mode %d", mode);
    }
}

// ------------------------------------------------------------------------------------------------
// Recurrent modules (Chain<Gru, Linear>)
// ------------------------------------------------------------------------------------------------
// RL_SEQ_FORCE_BIG=1 sends every size through the GEMM formulation (tests: K10 against K9 on the same small module)
bool seq_force_big() {
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("RL_SEQ_FORCE_BIG");
        v = (e && e[0] == '1') ? 1 : 0;
    }
    return v == 1;
}

// The shapes the recurrent passes are built for, on batches of F features (out_dim_expected > 0: that many outputs).
rl_status seq_check(rl_ctx *ctx, const rl_grunet_view &net, int F, int out_dim_expected, const char *what) {
    if (net.in_dim != F || (out_dim_expected > 0 && net.out_dim != out_dim_expected) ||
        !(rl_seq_pass_supports(net.in_dim, net.hidden, net.out_dim) || rl_seq_big_supports(net.in_dim, net.hidden, net.out_dim)))
        return rl_fail(ctx, RL_ERR_UNSUPPORTED, "%s: recurrent passes are built for hidden <= 128, features <= 64, outputs <= 32 "
                       "(got %d -> %d -> %d on %d features)", what, net.in_dim, net.hidden, net.out_dim, F);
    return RL_OK;
}

// ------------------------------------------------------------------------------------------------
// The module under update: an Mlp or a recurrent module, planned over one batch.  The algorithm drivers below see only
// its passes and its Adam step; which kind of module it is matters in init, pass and adam_step alone.
// ------------------------------------------------------------------------------------------------
// The batch of a trajectory: its planes over the time slots in use.
PassArgs traj_args(const rl_traj *traj) {
    PassArgs a{};
    a.obs = traj->obs; a.action = traj->action; a.succ = traj->succ;
    a.T = traj->used_T ? traj->used_T : traj->T;
    a.E = traj->E;
    return a;
}

struct UpdateNet {
    rl_ctx *ctx = nullptr;
    int P = 0;
    float *theta = nullptr;
    PassPlan plan{};
    char *extra = nullptr;  // the caller's extra_bytes of scratch
    PassArgs args{};        // batch, parameters and the update's inputs (adv, target, logp0, clip); vec and skip_flag per pass
    bool recurrent = false;
    PassNet pn{};            // an Mlp: which pass kernels
    rl_seq_pass_args seq{};  // a recurrent module: its shape and the scratch of back-propagation through time

    // An Mlp over `batch`; `logp0` reserves the behaviour log-probabilities of the batch after the caller's scratch.
    rl_status init(rl_ctx *c, rl_mlp *m, const PassNet &net, const PassArgs &batch, size_t extra_bytes, bool logp0) {
        ctx = c; P = (int)m->n_params; theta = m->params; pn = net;
        args = batch;
        args.theta = theta;
        const uint64_t TE = batch.T * batch.E;
        RL_TRY(make_plan(ctx, P, TE, &plan, extra_bytes + (logp0 ? TE * (size_t)pn.sh.A * sizeof(float) : 0), (void **)&extra));
        if (logp0) args.logp0 = (float *)(extra + extra_bytes);
        return RL_OK;
    }
    // A recurrent module over `batch`: one block of RL_SEQ_BLOCK lanes per partial row; after the caller's scratch, the
    // log-probabilities, the output cotangents and the hidden states of the batch (and an LSTM's cell states).
    rl_status init(rl_ctx *c, const rl_grunet_view &net, const PassArgs &batch, size_t extra_bytes) {
        ctx = c; P = (int)net.n_params; theta = net.params; recurrent = true;
        plan.P = P;
        plan.W = P + NSCALAR;
        plan.grid = (int)rl_div_up(batch.E, RL_SEQ_BLOCK);
        const size_t rows = (size_t)plan.grid * plan.W * sizeof(double), sums = ((size_t)plan.W * sizeof(double) + 255) / 256 * 256;
        const size_t TE = (size_t)batch.T * batch.E;
        const size_t lp = (TE * net.out_dim * sizeof(float) + 255) / 256 * 256, hb = (TE * net.hidden * sizeof(float) + 255) / 256 * 256;
        const size_t cb = net.cell == RL_CELL_LSTM ? hb : 0;
        extra_bytes = (extra_bytes + 255) / 256 * 256;
        char *buf;
        RL_TRY(rl_ctx_scratch(ctx, ((rows + 255) / 256 * 256) + sums + extra_bytes + 2 * lp + hb + cb + 256, (void **)&buf));
        plan.partials = (double *)buf;
        plan.sums = (double *)(buf + (rows + 255) / 256 * 256);
        extra = (char *)plan.sums + sums;
        args = batch;
        args.theta = theta;
        args.logp0 = (float *)(extra + extra_bytes);
        seq.F = net.in_dim; seq.H = net.hidden; seq.A = net.out_dim; seq.act = net.act; seq.cell = net.cell;
        seq.dzbuf = (float *)(extra + extra_bytes + lp);
        seq.hbuf = (float *)(extra + extra_bytes + 2 * lp);
        seq.cbuf = cb ? (float *)(extra + extra_bytes + 2 * lp + hb) : nullptr;
        seq.partials = plan.partials;
        return RL_OK;
    }

    // One full-batch pass in `mode`; leaves the all-reduced f64 sums in plan.sums.  A recurrent module's pass runs
    // gru_pass_kernel (K9), or K10's tiled GEMMs above its sizes.
    rl_status pass(int mode, const float *vec = nullptr, const int *skip_flag = nullptr) const {
        PassArgs a = args;
        a.vec = vec;
        a.skip_flag = skip_flag;
        if (!recurrent) return launch_pass_rt(ctx, plan, a, mode, pn);
        rl_seq_pass_args s = seq;
        s.obs = a.obs; s.action = a.action; s.succ = a.succ; s.T = a.T; s.E = a.E; s.theta = a.theta; s.vec = a.vec;
        s.adv = a.adv; s.target = a.target; s.logp0 = a.logp0; s.skip_flag = a.skip_flag;
        s.clip_lo = a.clip_lo; s.clip_hi = a.clip_hi;
        if (!rl_seq_pass_supports(s.F, s.H, s.A) || seq_force_big()) {
            // K10 (gru_big.cu): tiled GEMMs over the lanes of a step; one partial row
            RL_TRY(rl_seq_big_pass_launch(ctx, mode, s));
            return reduce_over_group(ctx, plan, 1, s.skip_flag);
        }
        RL_TRY(rl_seq_pass_launch(ctx, mode, s, plan.grid));
        return reduce_over_group(ctx, plan, plan.grid, s.skip_flag);
    }

    // One optimizer step on a pass in `mode`, its mean loss to *loss_out (n_backward_steps: zero_grad, backward, step;
    // torch/agents/mod.rs:50-55, coptimizer.rs:13-27).  An Mlp's pass leaves its rows to a kernel that reduces them (over
    // the peer mailboxes of the data-parallel group when they are mapped) and takes the step; a recurrent module's pass
    // is reduced as every pass is, then adam_step_kernel steps.
    rl_status adam_step(int mode, rl_adam *adam, const AdamArgs &ac, double *loss_out) const {
        if (recurrent) {
            RL_TRY(pass(mode));
            adam->step += 1;
            RL_LAUNCH(ctx, adam_step_kernel, 1, VEC_THREADS, 0, plan.sums, P, theta, adam->m, adam->v, ac, adam->step, loss_out);
            return RL_OK;
        }
        adam->step += 1;
        int rows = plan.grid;
        if (ctx->world > 1 && ctx->x_ok && rl_div_up(plan.W, 32) <= RL_X_BLOCKS) {
            RL_TRY(launch_pass_rt(ctx, plan, args, mode, pn, false, &rows));
            ctx->x_seq += 1;
            RL_LAUNCH(ctx, reduce_rows_x_kernel<true>, rl_div_up(plan.W, 32), 256, 0, plan.partials, rows, plan.W, plan.P, plan.sums,
                      ctx->x, ctx->x_seq, (const int *)nullptr, (XAdam{theta, adam->m, adam->v, ac, adam->step, loss_out, plan.P}));
        } else if (ctx->world > 1) {
            RL_TRY(launch_pass_rt(ctx, plan, args, mode, pn));
            RL_LAUNCH(ctx, adam_step_kernel, 1, VEC_THREADS, 0, plan.sums, plan.P, theta, adam->m, adam->v, ac, adam->step, loss_out);
        } else {
            RL_TRY(launch_pass_rt(ctx, plan, args, mode, pn, false, &rows));
            RL_LAUNCH(ctx, reduce_rows_adam_kernel, rl_div_up(plan.W, 32), 256, 0, plan.partials, rows, plan.W, plan.P, plan.sums,
                      theta, adam->m, adam->v, ac, adam->step, loss_out);
        }
        return RL_OK;
    }
};

// ------------------------------------------------------------------------------------------------
// The algorithm drivers and what they share
// ------------------------------------------------------------------------------------------------
// Device time of an update when the caller asked for statistics, on the context's two timing events (created on first
// use, freed by rl_ctx_destroy).
struct UpdateTimer {
    rl_ctx *ctx;
    bool on;
    rl_status start() {
        if (!on) return RL_OK;
        for (int k = 0; k < 2; ++k)
            if (!ctx->upd_ev[k]) RL_CUDA(ctx, cudaEventCreate(&ctx->upd_ev[k]));
        RL_CUDA(ctx, cudaEventRecord(ctx->upd_ev[0], ctx->stream));
        return RL_OK;
    }
    rl_status stop() {
        if (on) RL_CUDA(ctx, cudaEventRecord(ctx->upd_ev[1], ctx->stream));
        return RL_OK;
    }
    void elapsed(float *ms) const { cudaEventElapsedTime(ms, ctx->upd_ev[0], ctx->upd_ev[1]); }  // after a synchronisation
};

AdamArgs adam_args(const rl_adam *a) {
    return AdamArgs{a->cfg.learning_rate, a->cfg.beta1, a->cfg.beta2, a->cfg.weight_decay, a->cfg.eps};
}

// An optimizer for the n_params parameters of `owner` (the module's handle), moments at zero.
rl_status adam_create(rl_ctx *ctx, const void *owner, uint64_t n_params, const rl_adam_cfg *cfg, rl_adam **out, const char *what) {
    RL_CUDA(ctx, cudaSetDevice(ctx->device));
    rl_adam *a = new (std::nothrow) rl_adam();
    if (!a) return rl_fail(ctx, RL_ERR_OOM, "%s: host allocation failed", what);
    a->owner = owner;
    a->ctx = ctx;
    a->cfg = *cfg;
    cudaError_t e = cudaMalloc((void **)&a->m, n_params * sizeof(float));
    if (e == cudaSuccess) e = cudaMalloc((void **)&a->v, n_params * sizeof(float));
    if (e != cudaSuccess) {
        rl_adam_destroy(a);
        return rl_fail(ctx, RL_ERR_OOM, "%s: %s", what, cudaGetErrorString(e));
    }
    cudaMemsetAsync(a->m, 0, n_params * sizeof(float), ctx->stream);
    cudaMemsetAsync(a->v, 0, n_params * sizeof(float), ctx->stream);
    *out = a;
    return RL_OK;
}

// The checks of every Adam update: the optimizer was built for `module`, and the step count is in range.
rl_status adam_check(rl_ctx *ctx, const rl_adam *adam, const void *module, int n_steps, const char *what) {
    if (adam->owner != module) return rl_fail(ctx, RL_ERR_INVALID_ARG, "%s: optimizer belongs to another module", what);
    if (n_steps < 0 || n_steps > 100000) return rl_fail(ctx, RL_ERR_INVALID_ARG, "%s: optimizer steps out of range", what);
    return RL_OK;
}

// loss_first / loss_last of the n_steps losses (host), the sample count, the step count and the device time.
template <class Stats>
void fill_opt_stats(Stats *st, const double *losses, int n_steps, uint64_t num_steps, const UpdateTimer &timer) {
    st->loss_first = n_steps > 0 ? losses[0] : 0.0;
    st->loss_last = n_steps > 0 ? losses[n_steps - 1] : 0.0;
    st->num_steps = num_steps;
    st->opt_steps = (uint64_t)n_steps;
    timer.elapsed(&st->update_ms);
}

// One pass of `u` in `mode`, its sums read back to `host` (P parameter sums, then the SC_* scalars); with `loss` /
// `grad_host`, the mean loss and the flat gradient of the mean (sums over the pass's sample count).
rl_status probe_pass(const UpdateNet &u, int mode, const float *vec, std::vector<double> &host, double *loss, float *grad_host) {
    rl_ctx *ctx = u.ctx;
    RL_TRY(u.pass(mode, vec));
    host.resize((size_t)u.plan.W);
    RL_CUDA(ctx, cudaMemcpyAsync(host.data(), u.plan.sums, (size_t)u.plan.W * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const double N = host[u.P + SC_COUNT];
    if (loss) *loss = host[u.P + SC_LOSS] / N;
    if (grad_host)
        for (int i = 0; i < u.P; ++i) grad_host[i] = (float)(host[i] / N);
    return RL_OK;
}

// A P-vector of f32 in scratch, 256-byte aligned
size_t vec_bytes(int P) { return ((size_t)P * sizeof(float) + 255) / 256 * 256; }
size_t trpo_vector_bytes(int P) { return 256 + 6 * vec_bytes(P); }  // TrpoState + theta0, g, x, r, p, descent

// Trpo::update (trpo.rs:97-164) on the policy `u` (inputs: adv); u.extra holds trpo_vector_bytes.
rl_status trpo_update(const UpdateNet &u, const rl_trpo_cfg *cfg, rl_trpo_stats *stats, const char *what) {
    rl_ctx *ctx = u.ctx;
    const int P = u.P;
    const size_t vb = vec_bytes(P);
    const double *sums = u.plan.sums;
    float *theta = u.theta;
    char *ex = u.extra;
    TrpoState *st = (TrpoState *)ex;
    float *theta0 = (float *)(ex + 256), *g = (float *)(ex + 256 + vb), *x = (float *)(ex + 256 + 2 * vb);
    float *r = (float *)(ex + 256 + 3 * vb), *p = (float *)(ex + 256 + 4 * vb);
    float *descent = (float *)(ex + 256 + 5 * vb);
    UpdateTimer timer{ctx, stats != nullptr};
    RL_TRY(timer.start());
    const float reg = (float)cfg->hpv_reg_coeff;
    // behaviour-policy statistics (no_grad block, trpo.rs:112-122)
    RL_TRY(u.pass(RL_PASS_STATS));
    RL_LAUNCH(ctx, trpo_begin_kernel, 1, 32, 0, st, sums, P);
    // loss gradient at theta0 (conjugate_gradient.rs:121-143)
    RL_TRY(u.pass(RL_PASS_GRAD));
    RL_LAUNCH(ctx, trpo_cg_init_kernel, 1, VEC_THREADS, 0, st, sums, P, g, x, r, p, theta, theta0);
    // conjugate gradient on the Fisher matrix (conjugate_gradient.rs:371-403)
    for (uint64_t it = 0; it < cfg->cg_iterations; ++it) {
        RL_TRY(u.pass(RL_PASS_FVP, p, &st->cg_done));
        RL_LAUNCH(ctx, trpo_cg_step_kernel, 1, VEC_THREADS, 0, st, sums, P, x, r, p, reg, 1e-10);
    }
    RL_LAUNCH(ctx, trpo_nan_to_num_kernel, 1, VEC_THREADS, 0, st, x, P);
    RL_TRY(u.pass(RL_PASS_FVP, x));
    RL_LAUNCH(ctx, trpo_step_size_kernel, 1, VEC_THREADS, 0, st, sums, P, x, descent, reg, cfg->max_policy_step_kl);
    // backtracking line search (conjugate_gradient.rs:183-254)
    for (uint64_t i = 0; i < cfg->max_backtracks; ++i) {
        const double ratio = std::pow(cfg->backtrack_ratio, (double)i);
        RL_LAUNCH(ctx, trpo_ls_candidate_kernel, 1, VEC_THREADS, 0, st, theta, theta0, descent, (float)ratio, P);
        RL_TRY(u.pass(RL_PASS_EVAL, nullptr, &st->accepted));
        RL_LAUNCH(ctx, trpo_ls_check_kernel, 1, 32, 0, st, sums, P, cfg->max_policy_step_kl, (int)i, ratio);
    }
    RL_LAUNCH(ctx, trpo_ls_finish_kernel, 1, VEC_THREADS, 0, st, theta, theta0, P, cfg->max_policy_step_kl,
              cfg->accept_violation);
    TrpoState *host;
    RL_TRY(rl_ctx_pinned(ctx, sizeof(TrpoState), (void **)&host));
    RL_CUDA(ctx, cudaMemcpyAsync(host, st, sizeof(TrpoState), cudaMemcpyDeviceToHost, ctx->stream));
    RL_TRY(timer.stop());
    RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (stats) {
        stats->entropy = host->entropy; stats->step_size = host->step_size; stats->loss_initial = host->loss0;
        stats->loss_final = host->loss_final; stats->constraint_val_final = host->kl_final;
        stats->step_scale = host->step_scale; stats->num_backtracks = host->num_backtracks;
        stats->cg_iterations = host->cg_iters; stats->num_steps = (uint64_t)host->N;
        timer.elapsed(&stats->policy_update_ms);
    }
    const rl_status trpo_status = (rl_status)host->status;  // (x_error_check reuses the pinned scratch)
    RL_TRY(x_error_check(ctx, what));
    return trpo_status;
}

// Loss, KL and entropy of the policy `u` (inputs: adv) at its parameters, the flat gradient, and with a vector its
// Fisher-vector product plus hpv_reg_coeff times the vector; u.extra holds vec_bytes.
rl_status trpo_probe(const UpdateNet &u, const float *vec_host, double hpv_reg_coeff, double *loss, double *kl, double *entropy,
                     float *grad_host, float *fvp_host) {
    rl_ctx *ctx = u.ctx;
    const int P = u.P;
    std::vector<double> host;
    RL_TRY(probe_pass(u, RL_PASS_STATS, nullptr, host, nullptr, nullptr));
    const double N = host[P + SC_COUNT];
    if (entropy) *entropy = host[P + SC_ENTROPY] / N;
    RL_TRY(probe_pass(u, RL_PASS_GRAD, nullptr, host, loss, grad_host));
    if (kl) *kl = host[P + SC_KL] / N;
    if (vec_host && fvp_host) {
        float *vec = (float *)u.extra;
        RL_CUDA(ctx, cudaMemcpyAsync(vec, vec_host, (size_t)P * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
        RL_TRY(probe_pass(u, RL_PASS_FVP, vec, host, nullptr, nullptr));
        for (int i = 0; i < P; ++i) fvp_host[i] = (float)(host[i] / N) + vec_host[i] * (float)hpv_reg_coeff;
    }
    return RL_OK;
}

// ValuesOpt::update (opt.rs:100-127): n_steps Adam steps of the state-value module `u` (inputs: target) on the mean
// squared error; u.extra holds n_steps + 1 losses.
rl_status value_update(const UpdateNet &u, rl_adam *adam, int n_steps, rl_opt_stats *stats, const char *what) {
    rl_ctx *ctx = u.ctx;
    double *losses = (double *)u.extra;
    UpdateTimer timer{ctx, stats != nullptr};
    RL_TRY(timer.start());
    const AdamArgs ac = adam_args(adam);
    for (int s = 0; s < n_steps; ++s) RL_TRY(u.adam_step(RL_PASS_VALUE, adam, ac, losses + s));
    if (stats) {
        RL_TRY(timer.stop());
        double *host;
        RL_TRY(rl_ctx_pinned(ctx, (size_t)(n_steps + 4) * sizeof(double), (void **)&host));
        if (n_steps > 0) RL_CUDA(ctx, cudaMemcpyAsync(host, losses, (size_t)n_steps * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        RL_CUDA(ctx, cudaMemcpyAsync(host + n_steps, u.plan.sums + u.P + SC_COUNT, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        fill_opt_stats(stats, host, n_steps, n_steps > 0 ? (uint64_t)host[n_steps] : 0, timer);
    }
    return x_error_check(ctx, what);
}

// The losses of n_steps policy steps and [sum of entropies, N], 256-byte aligned
size_t policy_loss_bytes(int n_steps) { return ((size_t)(n_steps + 2) * sizeof(double) + 255) / 256 * 256; }

// Ppo::update (ppo.rs:97-147) with `ppo`, Reinforce::update (reinforce.rs:64-89) without, on the policy `u` (inputs: adv,
// logp0); u.extra holds policy_loss_bytes.
rl_status policy_adam_update(UpdateNet &u, rl_adam *adam, int n_steps, double clip_distance, bool ppo, rl_policy_opt_stats *stats,
                             const char *what) {
    rl_ctx *ctx = u.ctx;
    const double *sums = u.plan.sums;
    const int P = u.P;
    double *losses = (double *)u.extra;
    UpdateTimer timer{ctx, stats != nullptr};
    RL_TRY(timer.start());
    u.args.clip_lo = (float)(1.0 - clip_distance); u.args.clip_hi = (float)(1.0 + clip_distance);
    const AdamArgs ac = adam_args(adam);
    double *entropy_sum = losses + n_steps;  // [sum of entropies, N]
    if (ppo) {
        // initial log-probs and entropy under no_grad (ppo.rs:108-119)
        RL_TRY(u.pass(RL_PASS_STATS));
        RL_CUDA(ctx, cudaMemcpyAsync(entropy_sum, sums + P + SC_ENTROPY, sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
        RL_CUDA(ctx, cudaMemcpyAsync(entropy_sum + 1, sums + P + SC_COUNT, sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
        for (int s = 0; s < n_steps; ++s) RL_TRY(u.adam_step(RL_PASS_PPO, adam, ac, losses + s));
    } else {
        for (int s = 0; s < n_steps; ++s) {
            RL_TRY(u.adam_step(RL_PASS_REINFORCE, adam, ac, losses + s));
            if (s == 0) {  // entropies.get_or_insert_with: the distribution of the first loss evaluation (reinforce.rs:76)
                RL_CUDA(ctx, cudaMemcpyAsync(entropy_sum, sums + P + SC_ENTROPY, sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
                RL_CUDA(ctx, cudaMemcpyAsync(entropy_sum + 1, sums + P + SC_COUNT, sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
            }
        }
    }
    if (stats) {
        RL_TRY(timer.stop());
        double *host;
        RL_TRY(rl_ctx_pinned(ctx, (size_t)(n_steps + 4) * sizeof(double), (void **)&host));
        RL_CUDA(ctx, cudaMemcpyAsync(host, losses, (size_t)(n_steps + 2) * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        const bool have = ppo || n_steps > 0;
        fill_opt_stats(stats, host, n_steps, have ? (uint64_t)host[n_steps + 1] : 0, timer);
        stats->entropy = have && host[n_steps + 1] > 0 ? host[n_steps] / host[n_steps + 1] : 0.0;
    }
    return x_error_check(ctx, what);
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// C entry points: each checks its arguments, builds the UpdateNet of its module and runs the driver
// ------------------------------------------------------------------------------------------------
extern "C" {

void rl_trpo_cfg_default(rl_trpo_cfg *c) {
    // trpo.rs:29-38, conjugate_gradient.rs:55-64
    c->max_policy_step_kl = 0.01; c->cg_iterations = 10; c->max_backtracks = 15; c->backtrack_ratio = 0.8;
    c->hpv_reg_coeff = 1e-5; c->accept_violation = 0;
}

void rl_adam_cfg_default(rl_adam_cfg *c) {
    // coptimizer.rs:136-168; eps is libtorch's AdamOptions default
    c->learning_rate = 1e-3; c->beta1 = 0.9; c->beta2 = 0.999; c->weight_decay = 0.0; c->eps = 1e-8;
}

void rl_ppo_cfg_default(rl_ppo_cfg *c) {
    // ppo.rs:33-41
    c->opt_steps_per_update = 10;
    c->clip_distance = 0.2;
}

rl_status rl_pass_kernel_select(int32_t kernel) {
    if (kernel != RL_PASS_KERNEL_FFMA && kernel != RL_PASS_KERNEL_TCGEN05) return RL_ERR_INVALID_ARG;
    g_pass_kernel = kernel;
    return RL_OK;
}

rl_status rl_adam_create(rl_mlp *mlp, const rl_adam_cfg *cfg, rl_adam **out) {
    if (!mlp || !cfg || !out) return rl_fail(mlp ? mlp->ctx : nullptr, RL_ERR_INVALID_ARG, "rl_adam_create: NULL argument");
    return adam_create(mlp->ctx, mlp, mlp->n_params, cfg, out, "rl_adam_create");
}

rl_status rl_adam_create_seq(rl_grunet *net_h, const rl_adam_cfg *cfg, rl_adam **out) {
    if (!net_h || !cfg || !out) return rl_fail(nullptr, RL_ERR_INVALID_ARG, "rl_adam_create_seq: NULL argument");
    const rl_grunet_view net = rl_grunet_view_of(net_h);
    return adam_create(net.ctx, net_h, net.n_params, cfg, out, "rl_adam_create_seq");
}

rl_status rl_adam_destroy(rl_adam *a) {
    if (!a) return RL_OK;
    cudaSetDevice(a->ctx->device);
    cudaStreamSynchronize(a->ctx->stream);
    cudaFree(a->m); cudaFree(a->v);
    delete a;
    return RL_OK;
}

rl_status rl_trpo_update(rl_traj *traj, const float *adv_dev, rl_mlp *policy, const rl_trpo_cfg *cfg,
                         rl_trpo_stats *stats) {
    if (!traj || !adv_dev || !policy || !cfg)
        return rl_fail(traj ? traj->ctx : nullptr, RL_ERR_INVALID_ARG, "rl_trpo_update: NULL argument");
    rl_ctx *ctx = traj->ctx;
    PassNet pn;
    RL_TRY(pass_net_for(ctx, policy, (int)traj->F, "rl_trpo_update", &pn));
    UpdateNet u;
    RL_TRY(u.init(ctx, policy, pn, traj_args(traj), trpo_vector_bytes((int)policy->n_params), true));
    u.args.adv = adv_dev;
    return trpo_update(u, cfg, stats, "rl_trpo_update");
}

rl_status rl_trpo_update_seq(rl_traj *traj, const float *adv_dev, rl_grunet *policy, const rl_trpo_cfg *cfg,
                             rl_trpo_stats *stats) {
    if (!traj || !adv_dev || !policy || !cfg)
        return rl_fail(traj ? traj->ctx : nullptr, RL_ERR_INVALID_ARG, "rl_trpo_update_seq: NULL argument");
    rl_ctx *ctx = traj->ctx;
    const rl_grunet_view net = rl_grunet_view_of(policy);
    RL_REQUIRE(ctx, net.ctx == ctx, "rl_trpo_update_seq: module belongs to another context");
    RL_TRY(seq_check(ctx, net, (int)traj->F, 0, "rl_trpo_update_seq"));
    UpdateNet u;
    RL_TRY(u.init(ctx, net, traj_args(traj), trpo_vector_bytes((int)net.n_params)));
    u.args.adv = adv_dev;
    return trpo_update(u, cfg, stats, "rl_trpo_update_seq");
}

rl_status rl_trpo_probe(rl_traj *traj, const float *adv_dev, rl_mlp *policy, const float *vec_host, double hpv_reg_coeff,
                        double *loss, double *kl, double *entropy, float *grad_host, float *fvp_host) {
    if (!traj || !adv_dev || !policy) return rl_fail(traj ? traj->ctx : nullptr, RL_ERR_INVALID_ARG, "rl_trpo_probe: NULL argument");
    rl_ctx *ctx = traj->ctx;
    PassNet pn;
    RL_TRY(pass_net_for(ctx, policy, (int)traj->F, "rl_trpo_probe", &pn));
    UpdateNet u;
    RL_TRY(u.init(ctx, policy, pn, traj_args(traj), vec_bytes((int)policy->n_params), true));
    u.args.adv = adv_dev;
    return trpo_probe(u, vec_host, hpv_reg_coeff, loss, kl, entropy, grad_host, fvp_host);
}

rl_status rl_trpo_probe_seq(rl_traj *traj, const float *adv_dev, rl_grunet *policy, const float *vec_host,
                            double hpv_reg_coeff, double *loss, double *kl, double *entropy, float *grad_host,
                            float *fvp_host) {
    if (!traj || !adv_dev || !policy) return rl_fail(traj ? traj->ctx : nullptr, RL_ERR_INVALID_ARG, "rl_trpo_probe_seq: NULL argument");
    rl_ctx *ctx = traj->ctx;
    const rl_grunet_view net = rl_grunet_view_of(policy);
    RL_REQUIRE(ctx, net.ctx == ctx, "rl_trpo_probe_seq: module belongs to another context");
    RL_TRY(seq_check(ctx, net, (int)traj->F, 0, "rl_trpo_probe_seq"));
    UpdateNet u;
    RL_TRY(u.init(ctx, net, traj_args(traj), vec_bytes((int)net.n_params)));
    u.args.adv = adv_dev;
    return trpo_probe(u, vec_host, hpv_reg_coeff, loss, kl, entropy, grad_host, fvp_host);
}

rl_status rl_value_update(rl_traj *traj, const float *targets_dev, rl_mlp *value_fn, rl_adam *adam, int32_t n_steps,
                          rl_opt_stats *stats) {
    if (!traj || !targets_dev || !value_fn || !adam)
        return rl_fail(traj ? traj->ctx : nullptr, RL_ERR_INVALID_ARG, "rl_value_update: NULL argument");
    rl_ctx *ctx = traj->ctx;
    RL_TRY(adam_check(ctx, adam, value_fn, n_steps, "rl_value_update"));
    RL_REQUIRE(ctx, value_fn->out_dim == 1, "rl_value_update: a state-value module has one output");
    PassNet pn;
    RL_TRY(pass_net_for(ctx, value_fn, (int)traj->F, "rl_value_update", &pn));
    UpdateNet u;
    RL_TRY(u.init(ctx, value_fn, pn, traj_args(traj), (size_t)(n_steps + 1) * sizeof(double), false));
    u.args.target = targets_dev;
    return value_update(u, adam, n_steps, stats, "rl_value_update");
}

rl_status rl_value_update_seq(rl_traj *traj, const float *targets_dev, rl_grunet *value_fn, rl_adam *adam, int32_t n_steps,
                              rl_opt_stats *stats) {
    if (!traj || !targets_dev || !value_fn || !adam)
        return rl_fail(traj ? traj->ctx : nullptr, RL_ERR_INVALID_ARG, "rl_value_update_seq: NULL argument");
    rl_ctx *ctx = traj->ctx;
    const rl_grunet_view net = rl_grunet_view_of(value_fn);
    RL_REQUIRE(ctx, net.ctx == ctx, "rl_value_update_seq: module belongs to another context");
    RL_TRY(seq_check(ctx, net, (int)traj->F, 1, "rl_value_update_seq"));
    RL_TRY(adam_check(ctx, adam, value_fn, n_steps, "rl_value_update_seq"));
    UpdateNet u;
    RL_TRY(u.init(ctx, net, traj_args(traj), (size_t)(n_steps + 1) * sizeof(double)));
    u.args.target = targets_dev;
    return value_update(u, adam, n_steps, stats, "rl_value_update_seq");
}

rl_status rl_value_probe(rl_traj *traj, const float *targets_dev, rl_mlp *value_fn, int32_t kernel, double *loss,
                         float *grad_host) {
    if (!traj || !targets_dev || !value_fn) return rl_fail(traj ? traj->ctx : nullptr, RL_ERR_INVALID_ARG, "rl_value_probe: NULL argument");
    rl_ctx *ctx = traj->ctx;
    RL_REQUIRE(ctx, value_fn->out_dim == 1, "rl_value_probe: a state-value module has one output");
    PassNet pn;
    RL_TRY(pass_net_for(ctx, value_fn, (int)traj->F, "rl_value_probe", &pn));
    RL_REQUIRE(ctx, kernel == RL_PASS_KERNEL_FFMA || kernel == RL_PASS_KERNEL_TCGEN05, "rl_value_probe: unknown kernel");
    pn.kernel = kernel;
    UpdateNet u;
    RL_TRY(u.init(ctx, value_fn, pn, traj_args(traj), 0, false));
    u.args.target = targets_dev;
    std::vector<double> host;
    return probe_pass(u, RL_PASS_VALUE, nullptr, host, loss, grad_host);
}

rl_status rl_ppo_update(rl_traj *traj, const float *adv_dev, rl_mlp *policy, rl_adam *adam, const rl_ppo_cfg *cfg,
                        rl_policy_opt_stats *stats) {
    if (!traj || !adv_dev || !policy || !adam || !cfg)
        return rl_fail(traj ? traj->ctx : nullptr, RL_ERR_INVALID_ARG, "rl_ppo_update: NULL argument");
    rl_ctx *ctx = traj->ctx;
    const int n_steps = (int)cfg->opt_steps_per_update;
    RL_TRY(adam_check(ctx, adam, policy, n_steps, "rl_ppo_update"));
    PassNet pn;
    RL_TRY(pass_net_for(ctx, policy, (int)traj->F, "rl_ppo_update", &pn));
    UpdateNet u;
    RL_TRY(u.init(ctx, policy, pn, traj_args(traj), policy_loss_bytes(n_steps), true));
    u.args.adv = adv_dev;
    return policy_adam_update(u, adam, n_steps, cfg->clip_distance, true, stats, "rl_ppo_update");
}

rl_status rl_reinforce_update(rl_traj *traj, const float *adv_dev, rl_mlp *policy, rl_adam *adam, rl_policy_opt_stats *stats) {
    if (!traj || !adv_dev || !policy || !adam)
        return rl_fail(traj ? traj->ctx : nullptr, RL_ERR_INVALID_ARG, "rl_reinforce_update: NULL argument");
    rl_ctx *ctx = traj->ctx;
    RL_TRY(adam_check(ctx, adam, policy, 1, "rl_reinforce_update"));
    PassNet pn;
    RL_TRY(pass_net_for(ctx, policy, (int)traj->F, "rl_reinforce_update", &pn));
    UpdateNet u;
    RL_TRY(u.init(ctx, policy, pn, traj_args(traj), policy_loss_bytes(1), true));
    u.args.adv = adv_dev;
    return policy_adam_update(u, adam, 1, 0.0, false, stats, "rl_reinforce_update");
}

rl_status rl_ppo_update_seq(rl_traj *traj, const float *adv_dev, rl_grunet *policy, rl_adam *adam, const rl_ppo_cfg *cfg,
                            rl_policy_opt_stats *stats) {
    if (!traj || !adv_dev || !policy || !adam || !cfg)
        return rl_fail(traj ? traj->ctx : nullptr, RL_ERR_INVALID_ARG, "rl_ppo_update_seq: NULL argument");
    rl_ctx *ctx = traj->ctx;
    const rl_grunet_view net = rl_grunet_view_of(policy);
    RL_REQUIRE(ctx, net.ctx == ctx, "rl_ppo_update_seq: module belongs to another context");
    RL_TRY(seq_check(ctx, net, (int)traj->F, 0, "rl_ppo_update_seq"));
    const uint64_t n_steps = cfg->opt_steps_per_update;
    RL_TRY(adam_check(ctx, adam, policy, n_steps > 100000 ? -1 : (int)n_steps, "rl_ppo_update_seq"));
    UpdateNet u;
    RL_TRY(u.init(ctx, net, traj_args(traj), policy_loss_bytes((int)n_steps)));
    u.args.adv = adv_dev;
    return policy_adam_update(u, adam, (int)n_steps, cfg->clip_distance, true, stats, "rl_ppo_update_seq");
}

rl_status rl_reinforce_update_seq(rl_traj *traj, const float *adv_dev, rl_grunet *policy, rl_adam *adam, rl_policy_opt_stats *stats) {
    if (!traj || !adv_dev || !policy || !adam)
        return rl_fail(traj ? traj->ctx : nullptr, RL_ERR_INVALID_ARG, "rl_reinforce_update_seq: NULL argument");
    rl_ctx *ctx = traj->ctx;
    const rl_grunet_view net = rl_grunet_view_of(policy);
    RL_REQUIRE(ctx, net.ctx == ctx, "rl_reinforce_update_seq: module belongs to another context");
    RL_TRY(seq_check(ctx, net, (int)traj->F, 0, "rl_reinforce_update_seq"));
    RL_TRY(adam_check(ctx, adam, policy, 1, "rl_reinforce_update_seq"));
    UpdateNet u;
    RL_TRY(u.init(ctx, net, traj_args(traj), policy_loss_bytes(1)));
    u.args.adv = adv_dev;
    return policy_adam_update(u, adam, 1, 0.0, false, stats, "rl_reinforce_update_seq");
}

// DqnAgent::batch_update (dqn.rs:263-337) with an Mlp action-value module, on flat minibatch planes.
rl_status rl_dqn_update(rl_replay *rb, rl_mlp *q, rl_adam *adam, const rl_dqn_cfg *cfg, rl_opt_stats *stats) {
    if (!rb || !q || !adam || !cfg)
        return rl_fail(q ? q->ctx : nullptr, RL_ERR_INVALID_ARG, "rl_dqn_update: NULL argument");
    rl_ctx *ctx = rl_replay_ctx(rb);
    RL_REQUIRE(ctx, q->ctx == ctx, "rl_dqn_update: network belongs to another context");
    RL_TRY(adam_check(ctx, adam, q, cfg->opt_steps_per_update, "rl_dqn_update"));
    PassNet pn;
    RL_TRY(pass_net_for(ctx, q, rl_replay_num_features(rb), "rl_dqn_update", &pn));
    const size_t F = (size_t)pn.sh.F;
    const int n_steps = cfg->opt_steps_per_update;
    UpdateTimer timer{ctx, stats != nullptr};
    RL_TRY(timer.start());
    const AdamArgs ac = adam_args(adam);
    rl_minibatch_dev mb{};
    UpdateNet u;
    double *losses = nullptr;
    // sample_minibatch (dqn.rs:280-314): episodes, features and targets (no_grad) of every step.  Reward-to-go targets
    // do not depend on the parameters and the ring does not change during the update, so all n_steps minibatches are
    // sampled up front by three launches (identical to sampling them one by one); OneStepTd targets need the
    // parameters of their step and are sampled inside the loop.
    const bool batched = !cfg->target_one_step_td && n_steps > 1;
    if (batched)
        RL_TRY(rl_replay_sample_enqueue(rb, cfg->minibatch_steps, cfg->sample_seed, rl_replay_take_draw_indices(rb, (uint32_t)n_steps),
                                        0, cfg->discount_factor, q, (uint32_t)n_steps, &mb));
    for (int s = 0; s < n_steps; ++s) {
        if (!batched)
            RL_TRY(rl_replay_sample_enqueue(rb, cfg->minibatch_steps, cfg->sample_seed, rl_replay_next_draw_index(rb),
                                            cfg->target_one_step_td, cfg->discount_factor, q, 1, &mb));
        if (s == 0) {  // the minibatch planes hold at most minibatch_steps + one ring of columns: the plan is sized once
            PassArgs planes{};
            planes.T = 1;
            planes.E = mb.capacity;
            RL_TRY(u.init(ctx, q, pn, planes, (size_t)(n_steps + 1) * sizeof(double), false));
            losses = (double *)u.extra;
        }
        const size_t set = batched ? (size_t)s : 0;
        u.args.obs = mb.obs + set * mb.capacity * F; u.args.action = mb.action + set * mb.capacity;
        u.args.succ = mb.succ + set * mb.capacity; u.args.target = mb.target + set * mb.capacity;
        // loss_fn + backward_step (dqn.rs:316-336, coptimizer.rs:13-27)
        RL_TRY(u.adam_step(RL_PASS_QLOSS, adam, ac, losses + s));
    }
    uint64_t m_last = 0;
    if (n_steps > 0) RL_TRY(rl_replay_sample_finish(rb, &m_last, nullptr));
    if (stats) {
        RL_TRY(timer.stop());
        double *host;
        RL_TRY(rl_ctx_pinned(ctx, (size_t)(n_steps + 4) * sizeof(double), (void **)&host));
        if (n_steps > 0) RL_CUDA(ctx, cudaMemcpyAsync(host, losses, (size_t)n_steps * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        fill_opt_stats(stats, host, n_steps, m_last, timer);
    }
    return x_error_check(ctx, "rl_dqn_update");
}

// DqnAgent::batch_update (dqn.rs:263-337) with a recurrent action-value module: every optimizer step samples its episodes as
// sequences (rl_replay_sample_seq_dev: the draws of rl_dqn_update, one host read to size the planes), runs the Q-loss pass with
// back-propagation through time over them (K9 / K10), reduces over the data-parallel group and takes the Adam step.  One sample
// per optimizer step: the padded planes of a batched update could be opt_steps times B * L, far beyond the flat minibatches.
rl_status rl_dqn_update_seq(rl_replay *rb, rl_grunet *q, rl_adam *adam, const rl_dqn_cfg *cfg, rl_opt_stats *stats) {
    if (!rb || !q || !adam || !cfg)
        return rl_fail(rb ? rl_replay_ctx(rb) : nullptr, RL_ERR_INVALID_ARG, "rl_dqn_update_seq: NULL argument");
    rl_ctx *ctx = rl_replay_ctx(rb);
    const rl_grunet_view net = rl_grunet_view_of(q);
    RL_REQUIRE(ctx, net.ctx == ctx, "rl_dqn_update_seq: network belongs to another context");
    RL_TRY(adam_check(ctx, adam, q, cfg->opt_steps_per_update, "rl_dqn_update_seq"));
    RL_TRY(seq_check(ctx, net, rl_replay_num_features(rb), 0, "rl_dqn_update_seq"));
    const int n_steps = cfg->opt_steps_per_update;
    UpdateTimer timer{ctx, stats != nullptr};
    RL_TRY(timer.start());
    const AdamArgs ac = adam_args(adam);
    std::vector<double> losses((size_t)n_steps, 0.0);
    uint64_t m_last = 0;
    for (int s = 0; s < n_steps; ++s) {
        rl_traj *mb = nullptr;
        const float *target = nullptr;
        // sample_minibatch (dqn.rs:280-314); OneStepTd targets from the parameters of this step
        RL_TRY(rl_replay_sample_seq_dev(rb, cfg->minibatch_steps, cfg->sample_seed, rl_replay_next_draw_index(rb), cfg->target_one_step_td,
                                        cfg->discount_factor, q, &mb, &target));
        m_last = mb->num_steps;
        UpdateNet u;
        RL_TRY(u.init(ctx, net, traj_args(mb), 256));
        u.args.target = target;
        double *loss_dev = (double *)u.extra;
        // loss_fn + backward_step (dqn.rs:316-336, coptimizer.rs:13-27)
        RL_TRY(u.adam_step(RL_PASS_QLOSS, adam, ac, loss_dev));
        // the next sample synchronises anyway; the plan's scratch may move with the next sample's size
        if (stats) {
            RL_CUDA(ctx, cudaMemcpyAsync(&losses[(size_t)s], loss_dev, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
            RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        }
    }
    if (stats) {
        RL_TRY(timer.stop());
        RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        fill_opt_stats(stats, losses.data(), n_steps, m_last, timer);
    }
    return x_error_check(ctx, "rl_dqn_update_seq");
}

// One Q-loss pass of rl_dqn_update_seq for diagnostics and parity checks: the mean loss of the sequence minibatch of
// `draw_index` and its flat gradient at the current parameters (no Adam step).
rl_status rl_dqn_probe_seq(rl_replay *rb, const rl_dqn_cfg *cfg, rl_grunet *q, uint32_t draw_index, double *loss, float *grad_host) {
    if (!rb || !q || !cfg) return rl_fail(rb ? rl_replay_ctx(rb) : nullptr, RL_ERR_INVALID_ARG, "rl_dqn_probe_seq: NULL argument");
    rl_ctx *ctx = rl_replay_ctx(rb);
    const rl_grunet_view net = rl_grunet_view_of(q);
    RL_REQUIRE(ctx, net.ctx == ctx, "rl_dqn_probe_seq: network belongs to another context");
    RL_TRY(seq_check(ctx, net, rl_replay_num_features(rb), 0, "rl_dqn_probe_seq"));
    rl_traj *mb = nullptr;
    const float *target = nullptr;
    RL_TRY(rl_replay_sample_seq_dev(rb, cfg->minibatch_steps, cfg->sample_seed, draw_index, cfg->target_one_step_td, cfg->discount_factor,
                                    q, &mb, &target));
    UpdateNet u;
    RL_TRY(u.init(ctx, net, traj_args(mb), 0));
    u.args.target = target;
    std::vector<double> host;
    return probe_pass(u, RL_PASS_QLOSS, nullptr, host, loss, grad_host);
}

}  // extern "C"
