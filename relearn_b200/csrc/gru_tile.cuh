// gru_tile.cuh -- K8h: fused rollout with the rl2-sized recurrent policy (Chain<Gru(F -> 128), Linear(128 -> A)>,
// rl2-bandits.rs:379-393) where the GRU cell of a step is one register-tiled FP32 GEMM over the envs of a CTA.
// Included by gru.cu inside its anonymous namespace (uses GruView, SeqArgs and steps.cuh).
//
// Per step the cell is  [64 envs x (F + 128)] . [(F + 128) x 384]  (gate order r, z, n; libtorch gru_cell, see
// gru.cu) -- 1.1e5 FLOP per env-step, FP32-FMA bound (SURVEY 8d, K8).  K8a (one thread per env, hidden state in
// local memory) issues two loads per FMA; here
//   * a CTA owns 64 envs; the hidden state lives in shared memory as hs[unit][env] (double buffered), the
//     observation as xs[feature][env];
//   * the weights are kept once in global memory as Wt[F + 128][384] (k-major: row k holds column k of w_ih / w_hh
//     for all 384 gate units, built by gru_wt_kernel before the launch) and stream through a three-deep ring of
//     16-row chunks (24 KB) with cp.async.bulk + mbarrier complete_tx -- the 218 KB do not fit next to the state, and
//     one CTA-step needs them once per 3.5 M FMAs, so the stream costs ~7 B/clk of L2 bandwidth per SM;
//   * thread tile 8 envs x 4 units x 4 accumulators (r, z, input-n, hidden-n) as packed FFMA2: per k one row
//     costs 3 LDS.128 of weights + 2 LDS.128 of state for 48 FFMA2; a warp covers 16 units x all 64 envs so that a
//     quarter-warp touches 64 B of weights and 64 B of state per load (broadcast, conflict-free);
//   * epilogue in registers: r, z = sigmoid, n = tanh(in + r * hn), h' = (h - n) z + n, written to the other state
//     buffer (gates on the SFU: MUFU.EX2 + MUFU.RCP); then four threads per env fold relu(h') into the A logits
//     (FFMA2 over action pairs, two shuffles), and the env's owner thread samples the action, steps the env, stores
//     the step record and writes the next observation into xs.
// The owner's scalar state (env state, noise cursors, summary sums) lives in shared memory between steps so that the
// GEMM phase has the register file to itself.
// Measured (B200, 10 arms x 100 episodes, E = 18 944, T = 199): 337 M env-steps/s = 37.6 TFLOP/s = 56 % of the measured
// FMA peak; K8a: 12.4 M.  ncu: the GEMM loop is 70 % of the time at ~71 % of the FMA roof, co-limited by operand
// delivery (every LDS.128 moves 512 B into registers whatever the broadcast pattern: 160 shared-memory-pipe cycles per
// 192 FMA-pipe cycles per k).
#pragma once

constexpr int GT_H = 128, GT_N3 = 3 * GT_H;
constexpr int GT_MAXF = 32;
// Tile shapes: ENVS envs per CTA (4 threads per env), weight chunks of ROWS rows in a ring of NBUF buffers.
//   <64, 16, 3>: 256 threads, 185 KB of shared memory, one CTA per SM
//   <32, 8, 4>:  128 threads, 110 KB, two CTAs per SM -- one CTA's gate / sampling / env phase (few active lanes,
//                latency bound) overlaps the other's GEMM (FMA-pipe bound)
template <int ENVS, int ROWS, int NBUF>
struct GtShape {
    static constexpr int envs = ENVS, rows = ROWS, nbuf = NBUF, threads = 4 * ENVS;
    static constexpr int hld = ENVS + 4;       // row stride of hs (floats): 16-byte aligned rows, shifted banks
    static constexpr int ugw = 32 / (ENVS / 8);  // unit groups (of 4 units) per warp; a warp spans all ENVS envs
};

__device__ __forceinline__ void gt_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void gt_bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst), "l"(src),
                 "r"(bytes), "r"(bar)
                 : "memory");
}

// Gate nonlinearities on the SFU: exp2 (MUFU.EX2) and the approximate reciprocal (MUFU.RCP), ~2 ulp each; tanh as
// 2 sigmoid(2 x) - 1 (absolute error ~2e-7, no cancellation that matters: n enters h' additively).
__device__ __forceinline__ float gt_sigmoid(float v) { return __fdividef(1.0f, 1.0f + __expf(-v)); }
__device__ __forceinline__ float gt_tanh(float v) { return fmaf(2.0f, __fdividef(1.0f, 1.0f + __expf(-2.0f * v)), -1.0f); }

// Wt[k][g * H + j] = k < F ? w_ih[g * H + j][k] : w_hh[g * H + j][k - F]
__global__ void gru_wt_kernel(GruView m, float *__restrict__ wt) {
    const int N3 = 3 * m.H, total = (m.F + m.H) * N3;
    const float *w_ih = m.params, *w_hh = w_ih + (size_t)3 * m.H * m.F;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
        const int k = idx / N3, col = idx - k * N3;
        wt[idx] = k < m.F ? w_ih[(size_t)col * m.F + k] : w_hh[(size_t)col * m.H + (k - m.F)];
    }
}

template <class EnvT, bool REPLAY>
struct GtOwner {
    typename EnvT::State s;
    LaneNoise<REPLAY> nz;
    LaneStats st;
    float last_obs[EnvT::MAXF];
    uint32_t n, i;
    int succ_last, succ_prev;
};

constexpr int GT_LW = 16;  // row stride of the transposed Linear weights lin_w[unit][action]

template <class EnvT, bool REPLAY, class S>
constexpr size_t gt_smem_bytes() {
    return (size_t)S::nbuf * S::rows * GT_N3 * 4 + (size_t)2 * GT_H * S::hld * 4 + (size_t)GT_MAXF * S::envs * 4 +
           (size_t)GT_LW * GT_H * 4 + 4 * GT_H * 4 + 64 + S::envs * sizeof(GtOwner<EnvT, REPLAY>) + 64;
}

// EPS: the epsilon-greedy actor of a recurrent Q-network.  The cell runs for every env of the tile before the actor draws; an env
// whose actor explores copies its old state over the new one, so its hidden state does not advance (DqnActor::act, gru.cu).
template <class EnvT, bool REPLAY, class S, bool EPS>
__global__ void __launch_bounds__(S::threads, 256 / S::threads) rollout_seq_tile_kernel(typename EnvT::Params p, SeqArgs a) {
    constexpr int GT_ENVS = S::envs, GT_THREADS = S::threads, GT_ROWS = S::rows, GT_NBUF = S::nbuf, GT_HLD = S::hld;
    constexpr int MF = EnvT::MAXF, MA = EnvT::MAXA;
    static_assert(MA <= GT_LW && MA % 2 == 0, "actions are folded as FFMA2 pairs");
    using Owner = GtOwner<EnvT, REPLAY>;
    extern __shared__ __align__(128) unsigned char gt_smem[];
    float *ring = reinterpret_cast<float *>(gt_smem);                // [NBUF][ROWS][384]
    float *hs = ring + GT_NBUF * GT_ROWS * GT_N3;                    // [2][128][HLD]
    float *xs = hs + 2 * GT_H * GT_HLD;                              // [MAXF][64]
    float *lin_w = xs + GT_MAXF * GT_ENVS;                           // [128][GT_LW] (unit-major, zero padded)
    float *bias = lin_w + GT_LW * GT_H;                              // b_r, b_z, b_in, b_hn [128] each
    float *lin_b = bias + 4 * GT_H;                                  // [16]
    Owner *owners = reinterpret_cast<Owner *>(lin_b + 16);           // [64]
    uint64_t *bars = reinterpret_cast<uint64_t *>(owners + GT_ENVS);  // [NBUF]

    const int tid = threadIdx.x;
    const int F = a.F, A = a.A;
    const int nxc = (F + GT_ROWS - 1) / GT_ROWS;  // observation chunks per step
    const int cps = nxc + GT_H / GT_ROWS;         // chunks per step
    const uint32_t max_chunks = (a.min_steps ? a.min_steps + a.slack : 0) * (uint32_t)cps;

    {  // parameters that stay resident
        const float *b_ih = a.net.params + (size_t)3 * GT_H * F + (size_t)3 * GT_H * GT_H, *b_hh = b_ih + 3 * GT_H;
        const float *lw = b_hh + 3 * GT_H, *lb = lw + (size_t)A * GT_H;
        for (int j = tid; j < GT_H; j += GT_THREADS) {
            bias[j] = __fadd_rn(b_hh[j], b_ih[j]);
            bias[GT_H + j] = __fadd_rn(b_hh[GT_H + j], b_ih[GT_H + j]);
            bias[2 * GT_H + j] = b_ih[2 * GT_H + j];
            bias[3 * GT_H + j] = b_hh[2 * GT_H + j];
        }
        for (int j = tid; j < GT_LW * GT_H; j += GT_THREADS) {
            const int unit = j / GT_LW, k = j - unit * GT_LW;
            lin_w[j] = k < A ? lw[(size_t)k * GT_H + unit] : 0.0f;
        }
        if (tid < 16) lin_b[tid] = tid < A ? lb[tid] : 0.0f;
        for (int j = tid; j < 2 * GT_H * GT_HLD; j += GT_THREADS) hs[j] = 0.0f;  // SeqIterative::initial_state (gru.rs:23-28)
        for (int j = tid; j < GT_MAXF * GT_ENVS; j += GT_THREADS) xs[j] = 0.0f;
    }
    if (tid == 0) {
        for (int b = 0; b < GT_NBUF; ++b) tc::mbar_init(tc::smem_u32(&bars[b]), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }

    // chunk g of the stream: step-periodic, rows [r0, r0 + rows) of Wt into ring buffer g % NBUF
    auto issue = [&](uint32_t g) {
        const int c = (int)(g % (uint32_t)cps);
        const int r0 = c < nxc ? c * GT_ROWS : F + (c - nxc) * GT_ROWS;
        const int rows = c < nxc ? min(GT_ROWS, F - c * GT_ROWS) : GT_ROWS;
        const uint32_t b = g % GT_NBUF, bar = tc::smem_u32(&bars[b]), bytes = (uint32_t)rows * GT_N3 * 4u;
        gt_expect_tx(bar, bytes);
        gt_bulk_g2s(tc::smem_u32(ring + (size_t)b * GT_ROWS * GT_N3), a.wt + (size_t)r0 * GT_N3, bytes, bar);
    };

    // env owners: thread 4 e owns env e of the tile
    const int oe = tid >> 2, part = tid & 3;
    const bool owner = part == 0;
    const uint64_t e = (uint64_t)blockIdx.x * GT_ENVS + oe;
    const bool valid = e < a.E;
    const uint32_t t0 = a.noise.step_counter;
    Owner &o = owners[oe];
    auto observe_to_xs = [&]() {
        float obs[MF];
        EnvT::observe(p, o.s, obs);
#pragma unroll
        for (int f = 0; f < MF; ++f)
            if (f < F) xs[f * GT_ENVS + oe] = obs[f];
    };
    __syncthreads();
    if (owner) {
        o.st.init();
        o.i = 0;
        o.succ_last = o.succ_prev = RL_TERMINATE;
        o.n = (valid && a.min_steps) ? a.min_steps + a.slack : 0;  // take_steps.rs:20-31
#pragma unroll
        for (int f = 0; f < MF; ++f) o.last_obs[f] = 0.0f;
        if (valid) {
            o.nz.init(a.noise, a.lane_offset + e, e);
            if (o.n > 0) {  // train.rs:135: every period starts fresh episodes
                o.nz.set_step(t0);
                EnvT::template reset<REPLAY>(p, o.s, o.nz);
                observe_to_xs();
            }
        }
    }
    uint32_t g = 0, issued = 0;
    if (tid == 0)
        for (; issued < GT_NBUF && issued < max_chunks; ++issued) issue(issued);
    int any = __syncthreads_or(owner && o.n > 0);

    // GEMM tile of this thread: units u0 .. u0 + 3, envs e0 .. e0 + 7
    const int warp = tid >> 5, lane = tid & 31;
    const int u0 = 4 * S::ugw * warp + 4 * (lane % S::ugw), e0 = 8 * (lane / S::ugw);
    int cur = 0;
    while (any) {
        const float *hc = hs + (size_t)cur * GT_H * GT_HLD;
        float *hn = hs + (size_t)(cur ^ 1) * GT_H * GT_HLD;
        float2 accR[8][2], accZ[8][2], accI[8][2], accH[8][2];
        {
            const float4 br = *reinterpret_cast<const float4 *>(bias + u0), bz = *reinterpret_cast<const float4 *>(bias + GT_H + u0);
            const float4 bi = *reinterpret_cast<const float4 *>(bias + 2 * GT_H + u0), bh = *reinterpret_cast<const float4 *>(bias + 3 * GT_H + u0);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                accR[q][0] = make_float2(br.x, br.y); accR[q][1] = make_float2(br.z, br.w);
                accZ[q][0] = make_float2(bz.x, bz.y); accZ[q][1] = make_float2(bz.z, bz.w);
                accI[q][0] = make_float2(bi.x, bi.y); accI[q][1] = make_float2(bi.z, bi.w);
                accH[q][0] = make_float2(bh.x, bh.y); accH[q][1] = make_float2(bh.z, bh.w);
            }
        }
        for (int c = 0; c < cps; ++c, ++g) {
            const uint32_t b = g % GT_NBUF;
            tc::mbar_wait(tc::smem_u32(&bars[b]), (g / GT_NBUF) & 1u);
            const float *wb = ring + (size_t)b * GT_ROWS * GT_N3 + u0;
            if (c < nxc) {
                const int rows = min(GT_ROWS, F - c * GT_ROWS);
                const float *src = xs + (size_t)c * GT_ROWS * GT_ENVS + e0;
                for (int r = 0; r < rows; ++r) {
                    const float4 wr = *reinterpret_cast<const float4 *>(wb + r * GT_N3);
                    const float4 wz = *reinterpret_cast<const float4 *>(wb + r * GT_N3 + GT_H);
                    const float4 wn = *reinterpret_cast<const float4 *>(wb + r * GT_N3 + 2 * GT_H);
                    const float4 va = *reinterpret_cast<const float4 *>(src + r * GT_ENVS);
                    const float4 vb = *reinterpret_cast<const float4 *>(src + r * GT_ENVS + 4);
                    const float v[8] = {va.x, va.y, va.z, va.w, vb.x, vb.y, vb.z, vb.w};
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        const float2 vv = make_float2(v[q], v[q]);
                        accR[q][0] = __ffma2_rn(make_float2(wr.x, wr.y), vv, accR[q][0]);
                        accR[q][1] = __ffma2_rn(make_float2(wr.z, wr.w), vv, accR[q][1]);
                        accZ[q][0] = __ffma2_rn(make_float2(wz.x, wz.y), vv, accZ[q][0]);
                        accZ[q][1] = __ffma2_rn(make_float2(wz.z, wz.w), vv, accZ[q][1]);
                        accI[q][0] = __ffma2_rn(make_float2(wn.x, wn.y), vv, accI[q][0]);
                        accI[q][1] = __ffma2_rn(make_float2(wn.z, wn.w), vv, accI[q][1]);
                    }
                }
            } else {
                const float *src = hc + (size_t)(c - nxc) * GT_ROWS * GT_HLD + e0;
#pragma unroll
                for (int r = 0; r < GT_ROWS; ++r) {
                    const float4 wr = *reinterpret_cast<const float4 *>(wb + r * GT_N3);
                    const float4 wz = *reinterpret_cast<const float4 *>(wb + r * GT_N3 + GT_H);
                    const float4 wn = *reinterpret_cast<const float4 *>(wb + r * GT_N3 + 2 * GT_H);
                    const float4 va = *reinterpret_cast<const float4 *>(src + r * GT_HLD);
                    const float4 vb = *reinterpret_cast<const float4 *>(src + r * GT_HLD + 4);
                    const float v[8] = {va.x, va.y, va.z, va.w, vb.x, vb.y, vb.z, vb.w};
#pragma unroll
                    for (int q = 0; q < 8; ++q) {
                        const float2 vv = make_float2(v[q], v[q]);
                        accR[q][0] = __ffma2_rn(make_float2(wr.x, wr.y), vv, accR[q][0]);
                        accR[q][1] = __ffma2_rn(make_float2(wr.z, wr.w), vv, accR[q][1]);
                        accZ[q][0] = __ffma2_rn(make_float2(wz.x, wz.y), vv, accZ[q][0]);
                        accZ[q][1] = __ffma2_rn(make_float2(wz.z, wz.w), vv, accZ[q][1]);
                        accH[q][0] = __ffma2_rn(make_float2(wn.x, wn.y), vv, accH[q][0]);
                        accH[q][1] = __ffma2_rn(make_float2(wn.z, wn.w), vv, accH[q][1]);
                    }
                }
            }
            __syncthreads();  // every thread is done with ring buffer b
            if (tid == 0 && issued < max_chunks) {
                issue(issued);
                ++issued;
            }
        }
        // gates and the new hidden state (gru.cu header: libtorch gru_cell); unit-major so that the state moves as float4
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const float *hrow = hc + (size_t)(u0 + u) * GT_HLD + e0;
            const float4 ha = *reinterpret_cast<const float4 *>(hrow), hb = *reinterpret_cast<const float4 *>(hrow + 4);
            const float hold[8] = {ha.x, ha.y, ha.z, ha.w, hb.x, hb.y, hb.z, hb.w};
            float hnew[8];
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const float2 cr = accR[q][u >> 1], cz = accZ[q][u >> 1], ci = accI[q][u >> 1], ch = accH[q][u >> 1];
                const float r = gt_sigmoid(u & 1 ? cr.y : cr.x);
                const float z = gt_sigmoid(u & 1 ? cz.y : cz.x);
                const float n = gt_tanh(__fadd_rn(u & 1 ? ci.y : ci.x, __fmul_rn(u & 1 ? ch.y : ch.x, r)));
                hnew[q] = __fadd_rn(__fmul_rn(__fsub_rn(hold[q], n), z), n);
            }
            float *nrow = hn + (size_t)(u0 + u) * GT_HLD + e0;
            *reinterpret_cast<float4 *>(nrow) = make_float4(hnew[0], hnew[1], hnew[2], hnew[3]);
            *reinterpret_cast<float4 *>(nrow + 4) = make_float4(hnew[4], hnew[5], hnew[6], hnew[7]);
        }
        __syncthreads();
        // Linear over activation(h'): thread (env oe, part) folds units part, part + 4, ...
        float2 zp[MA / 2];
#pragma unroll
        for (int k = 0; k < MA / 2; ++k) zp[k] = make_float2(0.0f, 0.0f);
#pragma unroll 4
        for (int j = part; j < GT_H; j += 4) {
            const float av = rl_activate(a.net.act, hn[(size_t)j * GT_HLD + oe]);
            const float2 av2 = make_float2(av, av);
            const float4 *wrow = reinterpret_cast<const float4 *>(lin_w + j * GT_LW);
#pragma unroll
            for (int k4 = 0; k4 < (MA + 3) / 4; ++k4) {
                const float4 w4 = wrow[k4];
                zp[2 * k4] = __ffma2_rn(make_float2(w4.x, w4.y), av2, zp[2 * k4]);
                if (2 * k4 + 1 < MA / 2) zp[2 * k4 + 1] = __ffma2_rn(make_float2(w4.z, w4.w), av2, zp[2 * k4 + 1]);
            }
        }
        float zl[MA];
#pragma unroll
        for (int k = 0; k < MA; ++k) {
            zl[k] = k & 1 ? zp[k >> 1].y : zp[k >> 1].x;
            zl[k] += __shfl_xor_sync(0xffffffffu, zl[k], 1);
            zl[k] += __shfl_xor_sync(0xffffffffu, zl[k], 2);
            zl[k] += lin_b[k];
        }
        if (owner && o.n > 0) {
            const uint32_t i = o.i;
            o.nz.set_step(t0 + i);
            uint32_t action;
            if (EPS) {
                if (dqn_explore<REPLAY>(a, o.nz, A, action)) {
                    for (int j = 0; j < GT_H; ++j) hn[(size_t)j * GT_HLD + oe] = hc[(size_t)j * GT_HLD + oe];
                } else {
                    action = argmax_first<MA>(zl, A);
                }
            } else {
                const float u = rl_u32_to_f32(o.nz.template next_u32<RL_STREAM_ACTOR>());
                action = categorical_sample<MA>(zl, A, u);
            }
#pragma unroll
            for (int f = 0; f < MF; ++f)
                if (f < F) {
                    const float v = xs[f * GT_ENVS + oe];
                    a.obs[((uint64_t)i * F + f) * a.E + e] = v;
                    o.last_obs[f] = v;
                }
            float r;
            const int sc = EnvT::template step<REPLAY>(p, o.s, action, o.nz, r);
            if (sc == RL_INTERRUPT) {
                float obs[MF];
                EnvT::observe(p, o.s, obs);
#pragma unroll
                for (int f = 0; f < MF; ++f)
                    if (f < F) a.next_obs[((uint64_t)i * F + f) * a.E + e] = obs[f];
            }
            if (sc != RL_CONTINUE) {
                o.nz.set_step(t0 + i + 1);
                EnvT::template reset<REPLAY>(p, o.s, o.nz);
                for (int j = 0; j < GT_H; ++j) hn[(size_t)j * GT_HLD + oe] = 0.0f;  // steps.rs:116-124: actor.initial_state
            }
            observe_to_xs();
            a.action[(uint64_t)i * a.E + e] = (uint8_t)action;
            a.reward[(uint64_t)i * a.E + e] = r;
            a.succ[(uint64_t)i * a.E + e] = (uint8_t)sc;
            o.st.push(r, sc);
            o.succ_prev = o.succ_last;
            o.succ_last = sc;
            o.i = i + 1;
            uint32_t n = o.n - 1;
            if (sc != RL_CONTINUE && n <= a.slack) n = 0;  // take_steps.rs:83-88
            o.n = n;
        }
        any = __syncthreads_or(owner && o.n > 0);
        cur ^= 1;
    }
    // chunks already in flight must land before the CTA may exit
    for (; g < issued; ++g) tc::mbar_wait(tc::smem_u32(&bars[g % GT_NBUF]), (g / GT_NBUF) & 1u);

    LaneStats st;
    st.init();
    if (owner && valid) {
        st = o.st;
        const LaneEnd end = finalize_last_episode(o.i, o.succ_last, o.succ_prev);
        if (end.flags & 1u) a.succ[(uint64_t)end.len * a.E + e] = RL_PAD;
        if (end.flags & 2u) {
            a.succ[(uint64_t)(end.len - 1) * a.E + e] = RL_INTERRUPT;
#pragma unroll
            for (int f = 0; f < MF; ++f)
                if (f < F) a.next_obs[((uint64_t)(end.len - 1) * F + f) * a.E + e] = o.last_obs[f];
        }
        a.lane_len[e] = end.len;
        a.lane_flags[e] = (uint8_t)end.flags;
        st.set_stored(end);
        o.nz.finish(a.noise, e);
    }
    __syncthreads();  // xs is free now: it takes the block reduction's per-warp rows
    block_reduce_stats(st, owner && valid, reinterpret_cast<double (*)[ST_COUNT]>(xs), a.partials);
}

template <class EnvT, bool REPLAY, class S, bool EPS>
rl_status launch_seq_tile_k8h(rl_ctx *ctx, const typename EnvT::Params &p, SeqArgs &a) {
    const unsigned grid = (unsigned)((a.E + S::envs - 1) / S::envs);
    constexpr size_t smem = gt_smem_bytes<EnvT, REPLAY, S>();
    RL_CUDA(ctx, cudaFuncSetAttribute(rollout_seq_tile_kernel<EnvT, REPLAY, S, EPS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    RL_LAUNCH(ctx, (rollout_seq_tile_kernel<EnvT, REPLAY, S, EPS>), grid, S::threads, smem, p, a);
    return RL_OK;
}

template <class EnvT, class S>
rl_status launch_seq_tile_shape(rl_ctx *ctx, const typename EnvT::Params &p, SeqArgs &a, bool replay) {
    if (a.eps_greedy) {
        if (replay) return launch_seq_tile_k8h<EnvT, true, S, true>(ctx, p, a);
        return launch_seq_tile_k8h<EnvT, false, S, true>(ctx, p, a);
    }
    if (replay) return launch_seq_tile_k8h<EnvT, true, S, false>(ctx, p, a);
    return launch_seq_tile_k8h<EnvT, false, S, false>(ctx, p, a);
}

using GtWide = GtShape<64, 16, 3>;
using GtPair = GtShape<32, 8, 4>;

// tile_envs: 64 (the default) or 32 (two CTAs per SM; measured slower -- the two CTAs run in lockstep -- kept for tests)
template <class EnvT>
rl_status launch_seq_tile(rl_ctx *ctx, const typename EnvT::Params &p, SeqArgs &a, bool replay, int tile_envs) {
    if (tile_envs == 64) return launch_seq_tile_shape<EnvT, GtWide>(ctx, p, a, replay);
    return launch_seq_tile_shape<EnvT, GtPair>(ctx, p, a, replay);
}
