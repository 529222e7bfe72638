// pass_tc.cuh -- the full-batch passes of the update (K5 policy, K6 critic) on the 5th-generation tensor cores
// (tcgen05 + TMEM).
//
// Same contract as mlp_pass_kernel<5, A, 4, MODE>: one f64 partial row [P + NSCALAR] per CTA holding the sums over
// this CTA's samples of the loss / KL / entropy, the sample count and the gradient (or Fisher-vector product) for
// the 5 -> 128 -> A ReLU networks of the reference's defaults: the critic (A = 1, mse_loss(V(obs), targets),
// critics/opt.rs:100-127) and the two-action policy (A = 2: TRPO statistics / loss+KL / gradient / Fisher-vector
// product, trpo.rs:112-144, conjugate_gradient.rs:312-338; PPO, ppo.rs:124-138; REINFORCE, reinforce.rs:72-79).
// The description below is for the critic; the policy differences are listed after it.
//
// Why this maps to tensor cores although K = 5: a CTA owns tiles of 128 samples, one sample per thread and
// per TMEM lane, and both batch-sized contractions become MMAs whose operands are built in shared memory:
//
//   MMA1  pre[128 samples x 128 units] = X[128 x 48] . W1e[48 x 128]            (3 x tcgen05.mma K = 16)
//         Every f32 value is cut into three bf16 pieces hi + mid + lo (truncation: exact, 8 + 8 + 8 bits), and
//         the 48 K-slots hold the six piece products that matter to f32 accuracy for the 5 features and the
//         bias:  hi.hi, hi.mid, mid.hi, mid.mid, hi.lo, lo.hi   (dropped: <= 2^-24 relative each).  bf16
//         products are exact in the f32 accumulator, so pre is an f32-accurate W1 x + b1.
//   epilogue 1 (thread = sample): tcgen05.ld the 128 pre-activations of the sample; only their SIGNS are used:
//         the 0/1 ReLU mask as bf16 (exact), two units per PRMT + LOP3, written back to shared memory.  One spare
//         K-slot of MMA1 adds -2^-120 to every pre-activation so that an exact +0 (a zero-initialised unit)
//         counts as inactive, like relu'(0) = 0 in libtorch.
//   MMA3  Q[128 samples x 24] = Mask[128 x 128 units] . C[128 x 24],  c_jf = w2_j * [w1_j, b1_j]_f in four bf16 pieces
//         (8 x tcgen05.mma K = 16; the mask is the same bytes read K-major).  ReLU is piecewise linear, so
//         V_s = w2 . relu(pre_s) + b2 = sum_f [x_s, 1]_f * sum_j mask_sj c_jf + b2:
//         epilogue 3 needs 24 columns and 6 FMAs per sample instead of 128 max + 128 FMA.
//   epilogue 3: loss, dV = 2 (V - target), the six values y = dV * [x, 1] as 3 x bf16 pieces to shared memory.
//   MMA2  G[128 units x 18] = Mask^T[128 x 128 samples] . Y[128 x 18]              (8 x tcgen05.mma K = 16)
//         exact 0/1 times bf16 pieces, accumulated in TMEM (f32) over TC_DRAIN tiles, then in f64.
//
// The gradient follows from G_jf = sum_s mask_sj y_sf alone:
//   dW1[j][f] = w2_j G[j][f],  db1[j] = w2_j G[j][5],
//   dW2[j] = sum_s dV_s relu(pre_sj) = sum_s dV_s mask_sj (b1_j + w1_j . x_s) = b1_j G[j][5] + sum_f w1_jf G[j][f],
// so no further cross-sample contraction is needed.
//
// Two-action policy: MMA3 has one 24-column block per logit (z_k = sum_f [x,1]_f sum_j mask_sj w2_kj [w1_j,b1_j]_f), and
// for the Fisher-vector product a third block for the difference of the tangent logits, whose matrix is
// (v2_0 - v2_1)_j [w1_j,b1_j] + (w2_0 - w2_1)_j [v1_j,vb1_j] (forward tangent of a piecewise-linear net, same mask).
// Every per-sample logit gradient of a softmax sums to zero over the actions, so with two actions dz_1 = -dz_0 and
// ONE block Y = dz_0 [x,1] gives both: dW1[j] = (w2_0j - w2_1j) G[j], dW2[0][j] = -dW2[1][j] = b1_j G[j][5] + w1_j . G[j].
//
// Shared-memory operand layout: the no-swizzle canonical UMMA layout, 8 x 16 B core matrices stored as
// [chunk of 8 elements along the thread-private dimension][row = thread][16 B], so every operand store is one
// conflict-free 16 B store per thread (a warp writes 512 contiguous bytes).
#pragma once

#include "tcgen05.cuh"

// One launch = one full-batch pass; grid <= TC_CTAS_PER_SM * SMs, block = 128, dynamic smem = tc::tc_smem(blocks).
template <int A, int MODE>
struct TcPass : PassMode<MODE> {
    // Y blocks of MMA2: one, except for the Q-loss, whose logit gradients do not sum to zero (only the taken action's
    // output has one): block k holds y where action == k
    static constexpr int YBLOCKS = MODE == RL_PASS_QLOSS ? 2 : 1;
    static constexpr int N2 = tc::tc_n2(YBLOCKS);
    static constexpr int D2_COLS = N2 <= 32 ? 32 : 64;
    static constexpr int CTAS_PER_SM = YBLOCKS == 1 ? tc::TC_CTAS_PER_SM : 2;  // 128 + 64 TMEM columns, 80 KB of shared memory
    static constexpr int BLOCKS = A;  // 24-column blocks of MMA3: one per logit; FVP: z_0 - z_1 and its tangent
    static constexpr int N3 = tc::tc_n3(BLOCKS);
    static constexpr int SMEM = tc::tc_smem(BLOCKS, YBLOCKS);
    static_assert((A == 1 && MODE == RL_PASS_VALUE) || (A == 2 && MODE != RL_PASS_VALUE),
                  "built for the critic and for the two-action policy / action-value network");
};

template <int A, int MODE>
__global__ void __launch_bounds__(tc::TC_THREADS, TcPass<A, MODE>::CTAS_PER_SM) mlp_pass_tc_kernel(PassArgs a) {
    using namespace tc;
    using K = TcPass<A, MODE>;
    constexpr int F = 5, H = 128, P = H * F + H + A * H + A, W = P + NSCALAR;
    constexpr int NF = F + 1;   // features + the bias input
    constexpr int NY = 3 * NF;  // 18 columns of Y / G: three bf16 pieces of six values
    constexpr int NC = 4 * NF;  // 24 columns per block of C / Q: four pieces (see the setup of C)
    constexpr bool FVP = K::FVP, BACKWARD = K::BACKWARD, IS_POLICY = K::IS_POLICY;
    constexpr int N3 = K::N3, YB = K::YBLOCKS, N2 = K::N2;
    constexpr int RED = tc_red(K::BLOCKS, YB);
    if (a.skip_flag && *a.skip_flag) return;
    extern __shared__ __align__(128) unsigned char smem[];
    unsigned char *sA1 = smem + TC_A1, *sB1 = smem + TC_B1, *sA2 = smem + TC_A2, *sB2 = smem + TC_B2, *sB3 = smem + tc_b3(YB);
    double *red = reinterpret_cast<double *>(smem + RED);
    uint32_t *tptr = reinterpret_cast<uint32_t *>(smem + RED + 512 + 32);
    const uint32_t bar1 = smem_u32(smem + RED + 512), bar2 = bar1 + 8, bar3 = bar1 + 16;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

    // ---- one-time setup: this thread's hidden unit -> row `tid` of the B operands of MMA1 and MMA3 ----
    const float *tw1 = a.theta, *tb1 = tw1 + H * F, *tw2 = tb1 + H, *tb2 = tw2 + A * H;
    float wrow[NF], w2j[A], b2[A];
#pragma unroll
    for (int f = 0; f < F; ++f) wrow[f] = tw1[tid * F + f];
    wrow[F] = tb1[tid];
#pragma unroll
    for (int k = 0; k < A; ++k) {
        w2j[k] = tw2[k * H + tid];
        b2[k] = tb2[k];
    }
    float vb2d = 0.0f;  // FVP: difference of the direction's output biases
    {
        uint32_t hi[NF], mid[NF], lo[NF], e[40];
#pragma unroll
        for (int f = 0; f < NF; ++f) split3(wrow[f], hi[f], mid[f], lo[f]);
#pragma unroll
        for (int k = 0; k < 40; ++k) {
            const int g = k / NF, f = k % NF;  // piece pairing: x [hi hi mid mid hi lo] . w [hi mid hi mid lo hi]
            e[k] = k == 6 * NF ? 0x83800000u   // -2^-120 against the bias input: +0 pre-activations become negative
                   : k > 6 * NF ? 0u : (g == 0 || g == 2 || g == 5) ? hi[f] : (g == 1 || g == 3) ? mid[f] : lo[f];
        }
        store_row<5>(sB1, tid, e);
    }
    {
        // C: block k holds w2_kj * [w1_j, b1_j] (logit k).  FVP: block 0 is z_0 - z_1 (all the softmax needs) and
        // block 1 its tangent along `vec`: (v2_0 - v2_1)_j [w1_j, b1_j] + (w2_0 - w2_1)_j [v1_j, vb1_j].
        // Four bf16 pieces per value: three of the rounded product and one of its exact rounding residual
        // (fma(a, b, -fl(a b))) -- the regrouped sum over units cancels more than w2 . relu(pre) does, so the
        // products carry ~32 bits; the fourth piece is free (N stays 32 / 48).
        uint32_t e[N3];
#pragma unroll
        for (int b = 0; b < K::BLOCKS; ++b) {
            float c[NF], cr[NF];
            if (!FVP || b == 0) {
                const float w2b = !FVP ? w2j[b] : w2j[0] - w2j[A > 1 ? 1 : 0];
#pragma unroll
                for (int f = 0; f < NF; ++f) {
                    c[f] = __fmul_rn(w2b, wrow[f]);
                    cr[f] = __fmaf_rn(w2b, wrow[f], -c[f]);
                }
            } else {
                const float *pw1 = a.vec, *pb1 = pw1 + H * F, *pw2 = pb1 + H, *pb2 = pw2 + A * H;
                const float v2d = pw2[tid] - pw2[(A > 1 ? H : 0) + tid], w2d = w2j[0] - w2j[A > 1 ? 1 : 0];
                vb2d = pb2[0] - pb2[A > 1 ? 1 : 0];
#pragma unroll
                for (int f = 0; f < NF; ++f) {
                    const double exact = (double)v2d * (double)wrow[f] + (double)w2d * (double)(f < F ? pw1[tid * F + (f < F ? f : 0)] : pb1[tid]);
                    c[f] = (float)exact;
                    cr[f] = (float)(exact - (double)c[f]);
                }
            }
#pragma unroll
            for (int f = 0; f < NF; ++f) {
                uint32_t rh, rm, rl;
                split3(c[f], e[b * NC + f], e[b * NC + NF + f], e[b * NC + 2 * NF + f]);
                split3(cr[f], rh, rm, rl);
                e[b * NC + 3 * NF + f] = rh;
            }
        }
#pragma unroll
        for (int k = K::BLOCKS * NC; k < N3; ++k) e[k] = 0u;
        store_row<N3 / 8>(sB3, tid, e);
    }
    // K-slots 40..47 of both MMA1 operands are zero: one shared chunk
    *reinterpret_cast<uint4 *>(smem + TC_Z + tid * 16) = make_uint4(0u, 0u, 0u, 0u);
    if (warp == 0) {
        tmem_alloc(smem_u32(tptr), 128);
        if (BACKWARD) tmem_alloc(smem_u32(tptr + 1), K::D2_COLS);
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    if (tid == 0) {
        mbar_init(bar1, 1);
        mbar_init(bar2, 1);
        mbar_init(bar3, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    fence_async_smem();
    fence_before();
    __syncthreads();
    fence_after();
    const uint32_t tmem_d1 = tptr[0], tmem_d2 = BACKWARD ? tptr[1] : 0u;
    const uint32_t lane_off = (uint32_t)(warp * 32) << 16;

    constexpr uint32_t IDESC1 = make_idesc(128, 128, false, false);  // X (K-major) . W1e (K-major)
    constexpr uint32_t IDESC2 = make_idesc(128, N2, true, true);     // Mask^T (MN-major) . Y (MN-major)
    constexpr uint32_t IDESC3 = make_idesc(128, N3, false, true);    // Mask (K-major) . C (MN-major)
    const uint32_t aA1 = smem_u32(sA1), aB1 = smem_u32(sB1), aA2 = smem_u32(sA2), aB2 = smem_u32(sB2), aB3 = smem_u32(sB3);

    const uint64_t TE = a.T * a.E, ntiles = (TE + 127) / 128;
    double G[BACKWARD ? YB * NY : 1], sc[NSCALAR], gb2_acc[YB];
#pragma unroll
    for (int n = 0; n < (BACKWARD ? YB * NY : 1); ++n) G[n] = 0.0;
#pragma unroll
    for (int k = 0; k < YB; ++k) gb2_acc[k] = 0.0;
#pragma unroll
    for (int k = 0; k < NSCALAR; ++k) sc[k] = 0.0;

    // position of this thread's sample, advanced by one grid stride per tile without divisions
    const uint64_t stride = (uint64_t)gridDim.x * 128, stride_t = stride / a.E, stride_e = stride - stride_t * a.E;
    uint64_t n_next = (uint64_t)blockIdx.x * 128 + tid, t_next = n_next / a.E, e_next = n_next - t_next * a.E;
    struct Staged {
        float x[F], tgt, adv;
        float2 lp0;
        uint8_t code, act;
    };
    auto load_next = [&](Staged &st) {  // raw loads only: nothing here waits for the data
        const bool in_range = n_next < TE;
        st.code = in_range ? __ldg(a.succ + n_next) : (uint8_t)RL_PAD;
#pragma unroll
        for (int f = 0; f < F; ++f) st.x[f] = in_range ? __ldg(a.obs + (t_next * F + f) * a.E + e_next) : 0.0f;
        st.tgt = (K::USES_TARGET && in_range) ? __ldg(a.target + n_next) : 0.0f;
        st.act = (K::USES_ACT && in_range) ? __ldg(a.action + n_next) : (uint8_t)0;
        st.adv = (K::USES_ADV && in_range) ? __ldg(a.adv + n_next) : 0.0f;
        st.lp0 = make_float2(0.0f, 0.0f);
        if (K::USES_LP0 && in_range) st.lp0 = __ldg(reinterpret_cast<const float2 *>(a.logp0) + n_next);
        n_next += stride;
        t_next += stride_t;
        e_next += stride_e;
        if (e_next >= a.E) {
            e_next -= a.E;
            t_next += 1;
        }
    };
    auto drain = [&](uint32_t parity) {
        // G of the tiles accumulated so far: wait for the last MMA2, read this unit's 18 columns, add in f64
        mbar_wait(bar2, parity);
        fence_after();
        uint32_t r[YB * NY];
        tmem_ld_cols<YB * NY>(tmem_d2 + lane_off, r);
#pragma unroll
        for (int n = 0; n < (BACKWARD ? YB * NY : 1); ++n) G[n] += (double)__uint_as_float(r[n]);
    };

    Staged nxt;
    load_next(nxt);
    uint32_t it = 0;
    for (uint64_t tile = blockIdx.x; tile < ntiles; tile += gridDim.x, ++it) {
        const bool valid = nxt.code != RL_PAD;
        float x[F];
#pragma unroll
        for (int f = 0; f < F; ++f) x[f] = valid ? nxt.x[f] : 0.0f;
        const float tgt = valid ? nxt.tgt : 0.0f, adv_s = valid ? nxt.adv : 0.0f;
        const float lp0[2] = {valid ? nxt.lp0.x : 0.0f, valid ? nxt.lp0.y : 0.0f};
        const int act_s = valid ? (int)nxt.act : 0;
        const bool drained = BACKWARD && it > 0 && it % TC_DRAIN == 0;
        if (drained) drain((it - 1) & 1u);

        // ---- A operand of MMA1: this sample's row of X (pieces of the 5 features and of the bias input 1) ----
        {
            uint32_t hi[NF], mid[NF], lo[NF], e[40];
#pragma unroll
            for (int f = 0; f < F; ++f) split3(x[f], hi[f], mid[f], lo[f]);
            hi[F] = valid ? 0x3F800000u : 0u;
            mid[F] = 0u;
            lo[F] = 0u;
#pragma unroll
            for (int k = 0; k < 40; ++k) {
                const int g = k / NF, f = k % NF;
                e[k] = k == 6 * NF ? hi[F] : k > 6 * NF ? 0u : (g == 0 || g == 1 || g == 4) ? hi[f] : (g == 2 || g == 3) ? mid[f] : lo[f];
            }
            store_row<5>(sA1, tid, e);
        }
        fence_async_smem();
        fence_before();
        __syncthreads();
        if (tid == 0) {
            fence_after();
#pragma unroll
            for (int k = 0; k < 3; ++k)  // K = 16 per instruction = two 8-element chunks; the last pairs chunk 4 with the zero chunk
                umma_bf16(tmem_d1, make_desc(aA1 + k * 2 * TC_CHUNK, k < 2 ? TC_CHUNK : TC_Z - TC_A1 - 4 * TC_CHUNK, 128),
                          make_desc(aB1 + k * 2 * TC_CHUNK, k < 2 ? TC_CHUNK : TC_Z - TC_B1 - 4 * TC_CHUNK, 128), IDESC1, k > 0);
            umma_commit(bar1);
        }
        load_next(nxt);  // in flight during the MMAs and the epilogues

        // ---- epilogue 1: signs of the pre-activations -> 0/1 mask (bf16), chunk = 8 units, row = sample ----
        mbar_wait(bar1, it & 1u);
        if (BACKWARD && it > 0 && !drained) mbar_wait(bar2, (it - 1) & 1u);  // MMA2 of the previous tile has read the mask and Y
        fence_after();
#pragma unroll 1
        for (int c = 0; c < 4; ++c) {
            uint32_t r[32];
            tmem_ld32(tmem_d1 + lane_off + c * 32, r);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                uint32_t m[4];
#pragma unroll
                for (int i = 0; i < 4; ++i) m[i] = relu_mask_bf16x2(r[q * 8 + 2 * i], r[q * 8 + 2 * i + 1]);
                *reinterpret_cast<uint4 *>(sA2 + (c * 4 + q) * TC_CHUNK + tid * 16) = make_uint4(m[0], m[1], m[2], m[3]);
            }
        }
        fence_async_smem();
        fence_before();
        __syncthreads();
        if (tid == 0) {
            fence_after();
#pragma unroll
            for (int k = 0; k < 8; ++k)  // 16 units per instruction; Q lands in the first N3 columns of the (consumed) D1
                umma_bf16(tmem_d1, make_desc(aA2 + k * 2 * TC_CHUNK, TC_CHUNK, 128), make_desc(aB3 + k * 256, 128, TC_CHUNK), IDESC3, k > 0);
            umma_commit(bar3);
        }

        // ---- epilogue 3: the network outputs of this sample, then the per-sample algebra ----
        mbar_wait(bar3, it & 1u);
        fence_after();
        float z[A], zdd = 0.0f;  // logits (or V); FVP: tangent of z_0 - z_1
        {
            uint32_t r[K::BLOCKS * NC];
            tmem_ld_cols<K::BLOCKS * NC>(tmem_d1 + lane_off, r);
#pragma unroll
            for (int b = 0; b < K::BLOCKS; ++b) {
                // sum_f [x, 1]_f * (sum_j mask_sj c_jf); the four piece sums are added smallest first
                auto q = [&](int f) {
                    return ((__uint_as_float(r[b * NC + 3 * NF + f]) + __uint_as_float(r[b * NC + 2 * NF + f])) +
                            __uint_as_float(r[b * NC + NF + f])) + __uint_as_float(r[b * NC + f]);
                };
                float acc = q(F);
#pragma unroll
                for (int f = 0; f < F; ++f) acc = fmaf(x[f], q(f), acc);
                if (!FVP) z[b] = acc + b2[b];
                else if (b == 0) z[0] = acc + (b2[0] - b2[A > 1 ? 1 : 0]);  // softmax([z_0 - z_1, 0]) = softmax(z)
                else zdd = acc + vb2d;
            }
            if (FVP && A > 1) z[A > 1 ? 1 : 0] = 0.0f;
        }
        float dz0 = 0.0f;  // d loss / d z_0 (two actions: d loss / d z_1 = -dz0)
        if (valid) {
            float loss_s = 0.0f, kl_s = 0.0f, ent_s = 0.0f;
            if (IS_POLICY) {
                float lp[A], p[A];
                log_softmax<A>(z, A, lp);
#pragma unroll
                for (int k = 0; k < A; ++k) p[k] = expf(lp[k]);
                // onehot_0 - p_0 without the cancellation of 1 - p_0 near saturation: p_0 + p_1 = 1
                const float d0 = act_s == 0 ? p[A > 1 ? 1 : 0] : -p[0];
                if (MODE == RL_PASS_STATS) {
                    // trpo.rs:112-122: log-probs of the behaviour policy and its entropy (categorical.rs:62-68)
#pragma unroll
                    for (int k = 0; k < A; ++k) ent_s -= fmaxf(lp[k], F32_LOWEST) * p[k];
                    reinterpret_cast<float2 *>(a.logp0)[tile * 128 + tid] = make_float2(lp[0], lp[A > 1 ? 1 : 0]);
                }
                if (MODE == RL_PASS_EVAL || MODE == RL_PASS_GRAD) {
                    // trpo.rs:129-144: ratio = exp(logp - logp0); loss = -mean(ratio * adv); KL(p0 || p)
                    const float lpa = act_s == 0 ? lp[0] : lp[A > 1 ? 1 : 0], lp0a = act_s == 0 ? lp0[0] : lp0[1];
                    const float ratio = expf(lpa - lp0a);
                    loss_s = -(ratio * adv_s);
#pragma unroll
                    for (int k = 0; k < A; ++k) kl_s += fmaxf(lp0[k] - lp[k], F32_LOWEST) * expf(lp0[k]);
                    if (MODE == RL_PASS_GRAD) dz0 = loss_s * d0;
                }
                if (MODE == RL_PASS_PPO) {
                    // ppo.rs:124-138, backward as libtorch (see sample_loss, passes.cuh)
                    const float lpa = act_s == 0 ? lp[0] : lp[A > 1 ? 1 : 0], lp0a = act_s == 0 ? lp0[0] : lp0[1];
                    const float ratio = expf(lpa - lp0a);
                    const float clipped = fminf(fmaxf(ratio, a.clip_lo), a.clip_hi);
                    const float t1 = ratio * adv_s, t2 = clipped * adv_s;
                    loss_s = -fminf(t1, t2);
                    const bool inside = ratio >= a.clip_lo && ratio <= a.clip_hi;
                    const float g = (inside || t1 < t2) ? -t1 : 0.0f;
                    dz0 = g * d0;
                }
                if (MODE == RL_PASS_REINFORCE) {
                    // reinforce.rs:72-79
                    const float lpa = act_s == 0 ? lp[0] : lp[A > 1 ? 1 : 0];
                    loss_s = -(lpa * adv_s);
#pragma unroll
                    for (int k = 0; k < A; ++k) ent_s -= fmaxf(lp[k], F32_LOWEST) * p[k];
                    dz0 = -adv_s * d0;
                }
                if (FVP) dz0 = p[0] * (p[A > 1 ? 1 : 0] * zdd);  // u = (diag p - p p^T) zdot with p_0 + p_1 = 1
            } else if (MODE == RL_PASS_QLOSS) {
                // dqn.rs:316-326: mse(Q(obs).gather(action), targets); dz0 is the gradient w.r.t. the TAKEN action's output
                const float diff = (act_s == 0 ? z[0] : z[A > 1 ? 1 : 0]) - tgt;
                loss_s = diff * diff;
                dz0 = 2.0f * diff;
            } else {
                // opt.rs:109-115: mse_loss(V(obs), targets, Mean)
                const float diff = z[0] - tgt;
                loss_s = diff * diff;
                dz0 = 2.0f * diff;
            }
            sc[SC_COUNT] += 1.0;
            sc[SC_LOSS] += (double)loss_s;
            sc[SC_KL] += (double)kl_s;
            sc[SC_ENTROPY] += (double)ent_s;
#pragma unroll
            for (int k = 0; k < YB; ++k) gb2_acc[k] += (YB == 1 || (act_s == 0) == (k == 0)) ? (double)dz0 : 0.0;
        }
        if (BACKWARD) {
            uint32_t hi[NF], mid[NF], lo[NF], e[N2];
#pragma unroll
            for (int f = 0; f < NF; ++f) {
                const float y = f < F ? dz0 * x[f < F ? f : 0] : dz0;
                split3(y, hi[f], mid[f], lo[f]);
            }
#pragma unroll
            for (int k = 0; k < N2; ++k) {
                const int blk = k / NY, g = (k % NY) / NF, f = k % NF;
                const uint32_t piece = g == 0 ? hi[f] : g == 1 ? mid[f] : lo[f];
                e[k] = k >= YB * NY ? 0u : (YB == 1 || (act_s == 0) == (blk == 0)) ? piece : 0u;  // Q-loss: block of the taken action
            }
            store_row<N2 / 8>(sB2, tid, e);
            fence_async_smem();
            fence_before();
            __syncthreads();
            if (tid == 0) {
                fence_after();
#pragma unroll
                for (int k = 0; k < 8; ++k)  // 16 samples per instruction = two 8-sample groups of 128 B
                    umma_bf16(tmem_d2, make_desc(aA2 + k * 256, 128, TC_CHUNK), make_desc(aB2 + k * 256, 128, TC_CHUNK), IDESC2,
                              (k > 0 || it % TC_DRAIN != 0) ? 1u : 0u);
                umma_commit(bar2);
            }
        } else {
            fence_before();
            __syncthreads();  // every thread has read Q before the next tile's MMA1 overwrites D1
        }
    }
    if (BACKWARD && it > 0) drain((it - 1) & 1u);

    // ---- this CTA's partial row ----
    double s_sc[NSCALAR];
#pragma unroll
    for (int k = 0; k < NSCALAR; ++k) s_sc[k] = warp_sum_f64(sc[k]);
    double s_g[YB];
#pragma unroll
    for (int k = 0; k < YB; ++k) s_g[k] = warp_sum_f64(gb2_acc[k]);
    if (lane == 0) {
#pragma unroll
        for (int k = 0; k < NSCALAR; ++k) red[warp * 8 + k] = s_sc[k];
#pragma unroll
        for (int k = 0; k < YB; ++k) red[warp * 8 + NSCALAR + k] = s_g[k];
    }
    fence_before();
    __syncthreads();
    double *row = a.partials + (size_t)blockIdx.x * W;
    if (BACKWARD && YB == 1) {
        double Gf[NF];
#pragma unroll
        for (int f = 0; f < NF; ++f) Gf[f] = (G[f] + G[NF + f]) + G[2 * NF + f];
        // d/dz_1 = -d/dz_0 (A = 2): hidden-layer gradients see w2_0 - w2_1, the two output rows are opposite
        const double wd = A > 1 ? (double)w2j[0] - (double)w2j[A > 1 ? 1 : 0] : (double)w2j[0];
        double gw2 = (double)wrow[F] * Gf[F];
#pragma unroll
        for (int f = 0; f < F; ++f) {
            row[tid * F + f] = wd * Gf[f];
            gw2 += (double)wrow[f] * Gf[f];
        }
        row[H * F + tid] = wd * Gf[F];
        row[H * F + H + tid] = gw2;
        if (A > 1) row[H * F + H + H + tid] = -gw2;
    } else if (BACKWARD) {
        // Q-loss: one G per output, dW1[j] = sum_k w2_kj G^k[j], dW2[k][j] = b1_j G^k[j][5] + w1_j . G^k[j]
        double gw1[NF];
#pragma unroll
        for (int f = 0; f < NF; ++f) gw1[f] = 0.0;
#pragma unroll
        for (int k = 0; k < YB; ++k) {
            double Gf[NF];
#pragma unroll
            for (int f = 0; f < NF; ++f) Gf[f] = (G[k * NY + f] + G[k * NY + NF + f]) + G[k * NY + 2 * NF + f];
            double gw2 = (double)wrow[F] * Gf[F];
#pragma unroll
            for (int f = 0; f < F; ++f) gw2 += (double)wrow[f] * Gf[f];
#pragma unroll
            for (int f = 0; f < NF; ++f) gw1[f] += (double)w2j[k < A ? k : 0] * Gf[f];
            row[H * F + H + k * H + tid] = gw2;
        }
#pragma unroll
        for (int f = 0; f < F; ++f) row[tid * F + f] = gw1[f];
        row[H * F + tid] = gw1[F];
    } else {
        for (int i = tid; i < P; i += TC_THREADS) row[i] = 0.0;
    }
    if (tid == 0) {
        if (BACKWARD) {
#pragma unroll
            for (int k = 0; k < YB; ++k) {
                const double g = ((red[NSCALAR + k] + red[8 + NSCALAR + k]) + red[16 + NSCALAR + k]) + red[24 + NSCALAR + k];
                row[P - A + k] = g;
                if (YB == 1 && A > 1) row[P - 1] = -g;
            }
        }
#pragma unroll
        for (int k = 0; k < NSCALAR; ++k) row[P + k] = ((red[k] + red[8 + k]) + red[16 + k]) + red[24 + k];
    }
    if (warp == 0) {
        fence_after();
        tmem_dealloc(tmem_d1, 128);
        if (BACKWARD) tmem_dealloc(tmem_d2, K::D2_COLS);
    }
}
