// rollout_ws5.cuh -- K2z: the warp-specialised CartPole rollout for few envs (E <= 16 per SM), and what it shares with
// K2q (rollout_ws6.cuh, included after this file).  Included by rollout.cu inside its anonymous namespace.
//
// K2c<8> (rollout.cu) has each warp carry 4 envs x 8 threads and issue BOTH halves of the step chain: the policy
// (obs -> hidden layer -> logit difference -> compare) and the f64 dynamics, the latter redundantly in all 8 threads of an
// env.  With few envs the period is that combined instruction stream.  K2z splits it by warp.  A CTA owns 16 envs and has
// six warps:
//  * four POLICY warps, 4 envs x 8 threads each, with exactly K2c<8>'s register-resident hidden layer;
//  * one DYNAMICS warp whose lane (env, a) steps env `env` with action `a` speculatively: both actions of 16 envs fill
//    the warp, so nothing is computed redundantly;
//  * one AUX warp that draws every Philox block: the actor's uniform of each step, as its logit-space threshold, and the
//    would-be reset state of each step.  It fills them WS_CHUNK steps at a time into WS_RING-step shared-memory rings,
//    up to WS_AHEAD steps ahead of the dynamics warp.  Progress is three counters in shared memory, not a barrier:
//    `prod` (steps filled, written by the aux warp), `cons` (the dynamics warp's iteration, posted every fourth) and
//    `done` (the dynamics loop is over).  The dynamics warp waits on `prod` every fourth iteration, the policy warps
//    before every fourth step's thresholds.
// Per step, each dynamics lane publishes ITS candidate's next row -- observation after the step or, if the step ends the
// episode, after the reset; would-be `active` flag; successor code -- BEFORE the action is known, into a double-buffered
// mailbox rows[step parity][action][env].  The policy warps pick the row of the action they sampled themselves, so the
// select (shuffles) that follows serves only the dynamics warp's own next step.  Further work leaves the dynamics warp:
//  * the step record's successor code and reward are stored by two idle threads of the env's policy group one iteration
//    later (the row carries the previous step's code), the observation / action by the others; only the post-step
//    observation of an Interrupt (once per max_steps) is stored by the dynamics warp, behind a vote taken at the loop top;
//  * episode statistics are integer counters (exact, converted once); the copies kept for finalize_last_episode are
//    read back from the trajectory after the CTA-wide barrier that ends the loops;
//  * the loop condition uses the vote of the PREVIOUS iteration (one idle iteration at the end instead of a vote ->
//    branch dependency in every iteration); the policy warps stop on a flag in the row.
// Per-phase clocks (scripts/ws_clocks.sh, profiles/r2_summary.md section 5) put the period on the dynamics warp's own
// instruction stream; warps map to the four sub-partitions by index, and the dynamics warp sits on warp 2, the aux warp
// on warp 5 (RolloutArgs::dyn_* / aux_*, set by launch_ws5).
// Barriers: 1 / 3 = row of an even / odd step published (dynamics arrives, policy syncs), 2 / 4 = action of an even / odd
// step published (policy arrives, dynamics syncs).  Two ids per direction because the dynamics warp publishes the row of
// step i + 1 BEFORE it waits for the action of step i: with one id its arrival could land in the phase of step i that a
// late policy warp has not joined yet (seen as a hang with two CTAs per SM).
// Same operations on the same operands as K2c<8> (summation order of the logits included): bit-identical trajectories
// and summaries (tests/test_gpu_envs.py).  Philox noise and the categorical actor only.
#pragma once

constexpr int ZK_ENVS = 16, ZK_THREADS = 192, ZK_SYNC = 160;  // 160: the policy and dynamics warps meet at the barriers
constexpr int WS_RING = 16, WS_CHUNK = 4, WS_AHEAD = 11;        // the aux warp's rings (K2z and K2q)

__device__ __forceinline__ void named_bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
__device__ __forceinline__ void named_bar_arrive(int id, int n) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); }

// Shared memory through explicit 32-bit shared-window addresses (ld.shared / st.shared): with generic pointers ptxas
// rematerialises the window base (S2UR SR_CgaCtaId + ULEA) inside the loops.
__device__ __forceinline__ float4 smem_ld4(uint32_t a) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(a));
    return v;
}
__device__ __forceinline__ void smem_st4(uint32_t a, float4 v) {
    asm volatile("st.shared.v4.f32 [%0], {%1, %2, %3, %4};" ::"r"(a), "f"(v.x), "f"(v.y), "f"(v.z), "f"(v.w) : "memory");
}
__device__ __forceinline__ double2 smem_ldd2(uint32_t a) {
    double2 v;
    asm volatile("ld.shared.v2.f64 {%0, %1}, [%2];" : "=d"(v.x), "=d"(v.y) : "r"(a));
    return v;
}
__device__ __forceinline__ void smem_std2(uint32_t a, double2 v) {
    asm volatile("st.shared.v2.f64 [%0], {%1, %2};" ::"r"(a), "d"(v.x), "d"(v.y) : "memory");
}
__device__ __forceinline__ float smem_ldf(uint32_t a) {
    float v;
    asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ uint32_t smem_ldu(uint32_t a) {
    uint32_t v;
    asm volatile("ld.volatile.shared.u32 %0, [%1];" : "=r"(v) : "r"(a));
    return v;
}
__device__ __forceinline__ void smem_stu(uint32_t a, uint32_t v) { asm volatile("st.volatile.shared.u32 [%0], %1;" ::"r"(a), "r"(v) : "memory"); }
__device__ __forceinline__ void smem_stf(uint32_t a, float v) { asm volatile("st.shared.f32 [%0], %1;" ::"r"(a), "f"(v) : "memory"); }

#ifdef RL_WS_CLOCKS  // measurement build only (scripts/ws_clocks.sh): per-phase clocks of the dynamics / policy loops of two CTAs
__device__ __forceinline__ long long ws_clk(double dep, uint32_t dep2) {
    long long c;
    asm volatile("mov.u64 %0, %%clock64;" : "=l"(c) : "d"(dep), "r"(dep2) : "memory");
    return c;
}
#define WS_CLK(var, dep, dep2) const long long var = ws_clk(dep, dep2)
#else
#define WS_CLK(var, dep, dep2)
#endif

struct ZkShared {
    float4 sw4[4 * GK_PAIRS];
    float tail[4 + GK_REM_TABLE_MAX];
    // rows[step parity][action taken in the previous step][env]: (x, x', theta, theta') | (remaining, flags, -, -)
    // flags: bit 0 this env takes the step, bit 1 stop, bit 2 the env took the previous step, bits 8.. its successor code
    float4 rows[2][2][ZK_ENVS][2];
    uint32_t act[2][ZK_ENVS];          // [step parity][env]
    float thr[WS_RING][ZK_ENVS];       // logit-space thresholds
    double2 slot[WS_RING][ZK_ENVS][2]; // would-be reset states (x, x') | (theta, theta')
    uint32_t prod, cons, done, pad;
};
#define ZK_OFF(member) ((uint32_t)offsetof(ZkShared, member))
constexpr uint32_t ZK_ACTIVE = 1u, ZK_STOP = 2u, ZK_PREV_ACTIVE = 4u;

__global__ void __launch_bounds__(ZK_THREADS, 2) rollout_cartpole_ws5_kernel(CartPoleEnv::Params p, RolloutArgs a) {
    using EnvT = CartPoleEnv;
    constexpr int LANES = 8, PPL = GK_PAIRS / LANES;
    constexpr unsigned FULL = 0xffffffffu;
    extern __shared__ __align__(16) unsigned char gk_smem[];
    ZkShared &sh = *reinterpret_cast<ZkShared *>(gk_smem);
    // (through a shuffle: ptxas otherwise rematerialises the window base at its uses in the loops)
    const uint32_t sb = __shfl_sync(FULL, (uint32_t)__cvta_generic_to_shared(gk_smem), 0);
    const bool rem_table = p.max_steps != 0 && p.max_steps < GK_REM_TABLE_MAX;
    stage_pair_weights(a.net, sh.sw4, sh.tail, p, rem_table ? (int)p.max_steps + 1 : 0);
    const uint32_t rem_addr = sb + ZK_OFF(tail) + 8;
    auto remaining_feature = [&](uint32_t r) {
        return p.max_steps == 0 ? 0.0f : rem_table ? smem_ldf(rem_addr + 4u * r) : (float)__ddiv_rn((double)r, (double)p.max_steps);
    };
    const int hw_warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const bool later_cta = (int)blockIdx.x >= a.sm_count;
    const int dyn_warp = later_cta ? a.dyn_second : a.dyn_first, aux_warp = later_cta ? a.aux_second : a.aux_first;
    const bool is_dyn = hw_warp == dyn_warp, is_aux = hw_warp == aux_warp;
    const int warp = hw_warp - (hw_warp > dyn_warp ? 1 : 0) - (hw_warp > aux_warp ? 1 : 0);  // policy warp index 0..3
    const uint64_t e_base = (uint64_t)blockIdx.x * ZK_ENVS;
    const uint32_t t0 = a.noise.step_counter;
    const uint64_t seed = a.noise.seed;
    const int F = a.F;
    const uint64_t FE = (uint64_t)F * a.E;
    const uint32_t cap = a.min_steps ? a.min_steps + a.slack : 0;  // no env takes more steps than this
    LaneStats st;
    st.init();
    bool contributes = false;
    uint32_t fin_steps = 0;                                      // dynamics lanes: what finalize_last_episode needs after the loops
    int fin_succ_last = RL_TERMINATE, fin_succ_prev = RL_TERMINATE;

    // ---- aux: one chunk = WS_CHUNK steps x 16 envs; lane = (env, half) handles steps k0 + 2 half + {0, 1} ----
    auto aux_fill = [&](uint32_t k0) {
        const int el = lane & 15, half = lane >> 4;
        const uint64_t eg = e_base + el, lg = a.lane_offset + (eg < a.E ? eg : 0);
#pragma unroll 1
        for (int j = 0; j < 2; ++j) {
            const uint32_t k = k0 + 2u * (uint32_t)half + (uint32_t)j;
            const uint32_t ring = k & (WS_RING - 1);
            uint32_t oa[4], o0[4], o1[4];
            // policies/actor.rs:42-55: the actor's uniform of step k as the logit-space threshold (rl_logit_threshold)
            rl_philox4x32_10((uint32_t)lg, (uint32_t)(lg >> 32), t0 + k, (uint32_t)RL_STREAM_ACTOR * 64u, (uint32_t)seed,
                             (uint32_t)(seed >> 32), oa);
            // cartpole.rs:103-115: four uniform draws in field order = blocks 0 (x, x') and 1 (theta, theta')
            rl_philox4x32_10((uint32_t)lg, (uint32_t)(lg >> 32), t0 + k, (uint32_t)RL_STREAM_ENV_RESET * 64u, (uint32_t)seed,
                             (uint32_t)(seed >> 32), o0);
            rl_philox4x32_10((uint32_t)lg, (uint32_t)(lg >> 32), t0 + k, (uint32_t)RL_STREAM_ENV_RESET * 64u + 1u, (uint32_t)seed,
                             (uint32_t)(seed >> 32), o1);
            smem_stf(sb + ZK_OFF(thr) + 4u * (ring * ZK_ENVS + el), rl_logit_threshold(rl_u32_to_f32(oa[0])));
            const double x = rl_u64_to_uniform((uint64_t)o0[0] | ((uint64_t)o0[1] << 32), p.reset_low, p.reset_scale);
            const double xd = rl_u64_to_uniform((uint64_t)o0[2] | ((uint64_t)o0[3] << 32), p.reset_low, p.reset_scale);
            const double th = rl_u64_to_uniform((uint64_t)o1[0] | ((uint64_t)o1[1] << 32), p.reset_low, p.reset_scale);
            const double thd = rl_u64_to_uniform((uint64_t)o1[2] | ((uint64_t)o1[3] << 32), p.reset_low, p.reset_scale);
            const uint32_t sa = sb + ZK_OFF(slot) + 32u * (ring * ZK_ENVS + el);
            smem_std2(sa, make_double2(x, xd));
            smem_std2(sa + 16, make_double2(th, thd));
        }
    };
    if (threadIdx.x == 0) { sh.prod = 0; sh.cons = 0; sh.done = 0; }
    if (is_aux) {
        aux_fill(0);
        aux_fill(WS_CHUNK);
    }
    __syncthreads();
    if (is_aux && lane == 0) smem_stu(sb + ZK_OFF(prod), 2 * WS_CHUNK);

    if (is_aux) {
        // ------------------------------ aux warp ------------------------------
        uint32_t k0 = 2 * WS_CHUNK;
        while (k0 <= cap + 1) {
            // slots of steps k0 - 16 .. k0 - 13 are reused: their readers (thresholds at iteration k, reset states at
            // k - 1) are done once the dynamics warp is at iteration >= k0 - 12
            uint32_t c = smem_ldu(sb + ZK_OFF(cons));
            bool over = false;
            while (k0 > c + WS_AHEAD) {
                if (smem_ldu(sb + ZK_OFF(done))) { over = true; break; }
                __nanosleep(64);
                c = smem_ldu(sb + ZK_OFF(cons));
            }
            if (over) break;
            aux_fill(k0);
            __threadfence_block();
            __syncwarp();
            k0 += WS_CHUNK;
            if (lane == 0) smem_stu(sb + ZK_OFF(prod), k0);
        }
    } else if (is_dyn) {
        // ------------------------------ dynamics warp: lane = (env el, action act) ------------------------------
        const int el = lane & 15, act = lane >> 4;
        const uint64_t e = e_base + el;
        const bool valid = e < a.E;
        const uint64_t e_safe = valid ? e : 0;
        const float rem_full = remaining_feature(p.max_steps);
        const uint32_t slot0 = sb + ZK_OFF(slot) + 32u * (uint32_t)el;
        const uint32_t my_row = sb + ZK_OFF(rows) + 512u * (uint32_t)act + 32u * (uint32_t)el;  // + 1024 * step parity
        const uint32_t act_addr = sb + ZK_OFF(act) + 4u * (uint32_t)el;                          // + 64 * step parity
        // the reset state of noise step t0 + k, from the ring the aux warp keeps ahead
        auto fresh_state = [&](uint32_t k, EnvT::State &f) {
            const uint32_t sa = slot0 + 512u * (k & (WS_RING - 1));
            const double2 lo = smem_ldd2(sa), hi = smem_ldd2(sa + 16);
            f.x = lo.x; f.xd = lo.y; f.th = hi.x; f.thd = hi.y;
            f.meta = 0x80000000u | p.max_steps;
        };
        EnvT::State s;
        s.x = s.xd = s.th = s.thd = 0.0;
        s.meta = 0x80000000u | p.max_steps;
        uint32_t n = (valid && a.min_steps) ? a.min_steps + a.slack : 0;
        float obs4 = 0.0f;
        {
            EnvT::State f;
            fresh_state(0, f);
            if (n > 0) { s = f; obs4 = rem_full; }
        }
        bool go = __any_sync(FULL, n > 0);  // loop condition, one iteration behind
        smem_st4(my_row, make_float4((float)s.x, (float)s.xd, (float)s.th, (float)s.thd));
        smem_st4(my_row + 16, make_float4(obs4, __uint_as_float((n > 0 ? ZK_ACTIVE : 0u) | (go ? 0u : ZK_STOP)), 0.0f, 0.0f));
        __syncwarp();
        named_bar_arrive(1, ZK_SYNC);                     // row of step 0
        uint32_t it = 0;                                  // loop counter (= step index of the envs still active)
        uint32_t i = 0, cur_len = 0, n_eps = 0;           // steps stored, length of the running episode, episodes ended
        unsigned long long sum_el = 0ull, sum_el2 = 0ull; // sum of episode lengths and of their squares
        int succ_last = RL_TERMINATE, succ_prev = RL_TERMINATE;
#ifdef RL_WS_CLOCKS
        long long ck[5] = {0, 0, 0, 0, 0};
#endif
        while (go) {
            WS_CLK(c0, s.x, it);
            const bool active = n > 0;
            const uint32_t r_now = s.meta & 0x7FFFFFFFu;
            // an Interrupt can only come from the step limit running out (step_limit.rs:202-223): known before the step
            const bool some_limit = __any_sync(FULL, active && p.max_steps != 0 && r_now == 1);
            if ((it & 3u) == 0u && lane == 0) smem_stu(sb + ZK_OFF(cons), it);
            if ((it & 3u) == 3u) {  // the reset states of steps it + 1 .. it + 4
                while (smem_ldu(sb + ZK_OFF(prod)) < it + 5u) { }
                asm volatile("fence.acq_rel.cta;" ::: "memory");
            }
            // this lane's world: the step with action `act`, then -- if it ends the episode -- the reset (steps.rs:116-124)
            EnvT::State cand = s;
            const int cand_sc = EnvT::step_fast(p, cand, (uint32_t)act);
            EnvT::State fresh;
            fresh_state(it + 1, fresh);
            const float rem_cont = remaining_feature(r_now > 0 ? r_now - 1 : 0);
            const bool cand_ended = cand_sc != RL_CONTINUE;
            EnvT::State nxt;
            nxt.x = cand_ended ? fresh.x : cand.x; nxt.xd = cand_ended ? fresh.xd : cand.xd;
            nxt.th = cand_ended ? fresh.th : cand.th; nxt.thd = cand_ended ? fresh.thd : cand.thd;
            nxt.meta = cand_ended ? fresh.meta : cand.meta;
            uint32_t n_cand = n;
            if (active) {
                n_cand = n - 1;
                if (cand_ended && n_cand <= a.slack) n_cand = 0;  // take_steps.rs:83-88
            }
            const uint32_t row_w = my_row + 1024u * ((it + 1u) & 1u);
            smem_st4(row_w, make_float4((float)nxt.x, (float)nxt.xd, (float)nxt.th, (float)nxt.thd));
            smem_st4(row_w + 16, make_float4(cand_ended ? rem_full : rem_cont,
                                           __uint_as_float((n_cand > 0 ? ZK_ACTIVE : 0u) | (active ? ZK_PREV_ACTIVE : 0u) | ((uint32_t)cand_sc << 8)),
                                           0.0f, 0.0f));
            __syncwarp();
            named_bar_arrive(1 + 2 * (int)((it + 1u) & 1u), ZK_SYNC);
            WS_CLK(c1, nxt.x + nxt.thd, n_cand);
            named_bar_sync(2 + 2 * (int)(it & 1u), ZK_SYNC);
            WS_CLK(c2, 0.0, 0u);
            const uint32_t action = smem_ldu(act_addr + 64u * (it & 1u));
            const int src = el + 16 * (int)action;
            s.th = __shfl_sync(FULL, nxt.th, src);
            s.thd = __shfl_sync(FULL, nxt.thd, src);
            s.x = __shfl_sync(FULL, nxt.x, src);
            s.xd = __shfl_sync(FULL, nxt.xd, src);
            s.meta = __shfl_sync(FULL, nxt.meta, src);
            const int sc = __shfl_sync(FULL, cand_sc, src);
            const uint32_t n_next = __shfl_sync(FULL, n_cand, src);
            WS_CLK(c3, s.x + s.th, n_next);
            if (some_limit) {  // rare (once per max_steps): the post-step observation of an Interrupt (remaining == 0)
                const double px = __shfl_sync(FULL, cand.x, src), pxd = __shfl_sync(FULL, cand.xd, src);
                const double pth = __shfl_sync(FULL, cand.th, src), pthd = __shfl_sync(FULL, cand.thd, src);
                const uint32_t pmeta = __shfl_sync(FULL, cand.meta, src);
                if (active && sc == RL_INTERRUPT && act == 0) {
                    const uint64_t io = (uint64_t)i * FE + e_safe;
                    a.next_obs[io] = (float)px;
                    a.next_obs[io + a.E] = (float)pxd;
                    a.next_obs[io + 2 * a.E] = (float)pth;
                    a.next_obs[io + 3 * a.E] = (float)pthd;
                    if (F > 4) a.next_obs[io + 4 * a.E] = remaining_feature(pmeta & 0x7FFFFFFFu);
                }
            }
            // episode statistics (summary.rs:198-216) as exact integer counters
            const bool ended = active && sc != RL_CONTINUE;
            i += active ? 1u : 0u;
            cur_len += active ? 1u : 0u;
            n_eps += ended ? 1u : 0u;
            sum_el += ended ? (unsigned long long)cur_len : 0ull;
            sum_el2 += ended ? (unsigned long long)cur_len * cur_len : 0ull;
            cur_len = ended ? 0u : cur_len;
            succ_prev = active ? succ_last : succ_prev;
            succ_last = active ? sc : succ_last;
            n = n_next;
            go = __any_sync(FULL, active);  // == the vote on n > 0 taken one iteration ago
            it += 1;
#ifdef RL_WS_CLOCKS
            const long long c4 = ws_clk((double)sum_el2, i + cur_len);
            ck[0] += c1 - c0; ck[1] += c2 - c1; ck[2] += c3 - c2; ck[3] += c4 - c3; ck[4] += 1;
#endif
        }
        if (it > 0) {
            // The policy warps have taken the rows of steps 0 .. it and wait for one more: tell them to stop, and take the
            // action they publish for step `it` (no env is active in steps it - 1 and it).
            const uint32_t row_w = my_row + 1024u * ((it + 1u) & 1u);
            smem_st4(row_w + 16, make_float4(0.0f, __uint_as_float(ZK_STOP), 0.0f, 0.0f));
            __syncwarp();
            named_bar_arrive(1 + 2 * (int)((it + 1u) & 1u), ZK_SYNC);
            named_bar_sync(2 + 2 * (int)(it & 1u), ZK_SYNC);
        }
#ifdef RL_WS_CLOCKS
        if (lane == 0 && ck[4] > 0 && (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1))
            printf("K2z dyn cta %d: %lld iterations; clk per iteration: candidate step + publish %.1f, wait for the action %.1f, "
                   "select %.1f, bookkeeping %.1f\n", (int)blockIdx.x, ck[4], (double)ck[0] / ck[4], (double)ck[1] / ck[4],
                   (double)ck[2] / ck[4], (double)ck[3] / ck[4]);
#endif
        if (lane == 0) smem_stu(sb + ZK_OFF(done), 1u);
        st.v[ST_STEPS] = st.v[ST_R] = st.v[ST_R2] = (double)i;
        st.v[ST_EPS] = (double)n_eps; st.v[ST_ER] = st.v[ST_EL] = (double)sum_el; st.v[ST_ER2] = st.v[ST_EL2] = (double)sum_el2;
        fin_steps = i; fin_succ_last = succ_last; fin_succ_prev = succ_prev;
    } else {
        // ------------------------------ policy warps: 4 envs x 8 threads (K2c<8>) ------------------------------
        const int grp = lane >> 3, sub = lane & 7, el = 4 * warp + grp;
        const uint64_t e = e_base + el;
        const bool valid = e < a.E;
        const uint64_t e_safe = valid ? e : 0;
        const float b2d = sh.tail[0];
        float4 wA[PPL], wB[PPL], wC[PPL];
        float2 wD[PPL];
#pragma unroll
        for (int u = 0; u < PPL; ++u) {
            const int q = sub + LANES * u;
            wA[u] = sh.sw4[q]; wB[u] = sh.sw4[GK_PAIRS + q]; wC[u] = sh.sw4[2 * GK_PAIRS + q];
            wD[u] = make_float2(sh.sw4[3 * GK_PAIRS + q].x, sh.sw4[3 * GK_PAIRS + q].y);
        }
        // Thread `sub` stores column `sub` of the step record: observation feature sub (< F), sub == 5 the action and, one
        // iteration later, sub == 6 the successor code and sub == 7 the reward.
        const bool stores_obs = valid && sub < 5 && sub < F, stores_action = valid && sub == 5;
        const bool stores_succ = valid && sub == 6, stores_reward = valid && sub == 7;
        float *obs_ptr = a.obs + (uint64_t)(sub < 5 ? sub : 0) * a.E + e_safe;
        uint8_t *act_ptr = a.action + e_safe;
        uint8_t *succ_ptr = a.succ + e_safe;     // of the previous step: one row behind (not dereferenced at i == 0)
        float *reward_ptr = a.reward + e_safe;
        const uint32_t row0 = sb + ZK_OFF(rows) + 32u * (uint32_t)el, mine_off = 4u * (uint32_t)(sub < 5 ? sub : 0);
        const uint32_t thr_addr = sb + ZK_OFF(thr) + 4u * (uint32_t)el, act_addr = sb + ZK_OFF(act) + 4u * (uint32_t)el;
        uint32_t prev_action = 0;
#ifdef RL_WS_CLOCKS
        long long pk[4] = {0, 0, 0, 0};
#endif
        for (uint32_t i = 0;; ++i) {
            WS_CLK(q0, 0.0, i);
            if ((i & 3u) == 0u) {  // thresholds of steps i .. i + 3
                // (`done`: the dynamics warp has left its loop and the aux warp may have stopped; this iteration only breaks)
                while (smem_ldu(sb + ZK_OFF(prod)) < i + 4u && !smem_ldu(sb + ZK_OFF(done))) { }
                asm volatile("fence.acq_rel.cta;" ::: "memory");
            }
            const float theta = smem_ldf(thr_addr + 64u * (i & (WS_RING - 1)));
            const uint32_t row = row0 + 1024u * (i & 1u) + 512u * prev_action;
            named_bar_sync(1 + 2 * (int)(i & 1u), ZK_SYNC);
            WS_CLK(q1, 0.0, 0u);
            const float4 ov = smem_ld4(row);
            const float4 tv = smem_ld4(row + 16);
            const float mine = smem_ldf(row + mine_off);
            const float ob4 = tv.x;
            const uint32_t flags = __float_as_uint(tv.y);
            // the previous step's successor code and reward (simulation/mod.rs PartialStep -> buffers/vec.rs)
            if ((flags & ZK_PREV_ACTIVE) != 0u) {
                if (stores_succ) *(succ_ptr - a.E) = (uint8_t)(flags >> 8);
                if (stores_reward) *(reward_ptr - a.E) = 1.0f;  // cartpole.rs:140
            }
#ifdef RL_WS_CLOCKS
            if ((flags & ZK_STOP) != 0u && warp == 0 && lane == 0 && pk[3] > 0 && (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1))
                printf("K2z policy cta %d: %lld iterations; clk per iteration: wait for the row %.1f, row -> action published %.1f, "
                       "record stores %.1f\n", (int)blockIdx.x, pk[3], (double)pk[0] / pk[3], (double)pk[1] / pk[3], (double)pk[2] / pk[3]);
#endif
            if ((flags & ZK_STOP) != 0u) break;
            const bool active = (flags & ZK_ACTIVE) != 0u;
            const float2 o0 = make_float2(ov.x, ov.x), o1 = make_float2(ov.y, ov.y), o2 = make_float2(ov.z, ov.z);
            const float2 o3 = make_float2(ov.w, ov.w), o4 = make_float2(ob4, ob4);
            float2 pre[PPL];
#pragma unroll
            for (int u = 0; u < PPL; ++u) pre[u] = __ffma2_rn(make_float2(wA[u].x, wA[u].y), o0, make_float2(wC[u].z, wC[u].w));
#pragma unroll
            for (int u = 0; u < PPL; ++u) pre[u] = __ffma2_rn(make_float2(wA[u].z, wA[u].w), o1, pre[u]);
#pragma unroll
            for (int u = 0; u < PPL; ++u) pre[u] = __ffma2_rn(make_float2(wB[u].x, wB[u].y), o2, pre[u]);
#pragma unroll
            for (int u = 0; u < PPL; ++u) pre[u] = __ffma2_rn(make_float2(wB[u].z, wB[u].w), o3, pre[u]);
#pragma unroll
            for (int u = 0; u < PPL; ++u) pre[u] = __ffma2_rn(make_float2(wC[u].x, wC[u].y), o4, pre[u]);
            float2 za = make_float2(0.0f, 0.0f), zc = make_float2(0.0f, 0.0f);
#pragma unroll
            for (int u = 0; u < PPL; ++u) {
                const float2 h = make_float2(fmaxf(pre[u].x, 0.0f), fmaxf(pre[u].y, 0.0f));
                if (u & 1) zc = __ffma2_rn(wD[u], h, zc);
                else za = __ffma2_rn(wD[u], h, za);
            }
            za = __fadd2_rn(za, zc);
            float d = za.x + za.y;
#pragma unroll
            for (int o = LANES / 2; o > 0; o >>= 1) d += __shfl_xor_sync(FULL, d, o);
            d += b2d;
            const uint32_t action = d < theta ? 0u : 1u;  // policies/actor.rs:42-55 (rl_logit_threshold)
            if (sub == 0) smem_stu(act_addr + 64u * (i & 1u), action);
            __syncwarp();
            named_bar_arrive(2 + 2 * (int)(i & 1u), ZK_SYNC);
            WS_CLK(q2, 0.0, action);
            // ---- off the chain: the observation and the action of the step record ----
            if (active && stores_obs) *obs_ptr = mine;
            if (active && stores_action) *act_ptr = (uint8_t)action;
            obs_ptr += FE;
            act_ptr += a.E;
            succ_ptr += a.E;
            reward_ptr += a.E;
            prev_action = action;
#ifdef RL_WS_CLOCKS
            const long long q3 = ws_clk(0.0, (uint32_t)(uintptr_t)act_ptr);
            pk[0] += q1 - q0; pk[1] += q2 - q1; pk[2] += q3 - q2; pk[3] += 1;
#endif
        }
    }
    __syncthreads();  // one barrier for every role: the policy warps' stores of the step records are visible from here on
    if (is_dyn) {
        const int act = lane >> 4;
        const uint64_t e = e_base + (lane & 15);
        if (e < a.E && act == 0) {
            // VecBuffer::end_experience -> finalize_last_episode (buffers/mod.rs:237-261), steps.cuh's rule spelled out: with
            // the helper, ptxas schedules the step loops above differently, and K2q's period was 0.3 % longer (B200, 1000 W)
            const uint32_t i = fin_steps;
            const int succ_last = fin_succ_last, succ_prev = fin_succ_prev;
            uint32_t len = i, flags = 0;
            double eps = st.v[ST_EPS];
            if (i > 0 && succ_last == RL_CONTINUE) {
                len = i - 1;
                flags = 1;
                a.succ[(uint64_t)len * a.E + e] = RL_PAD;
                if (len > 0 && succ_prev == RL_CONTINUE) {
                    flags = 3;
                    a.succ[(uint64_t)(len - 1) * a.E + e] = RL_INTERRUPT;
                    // next_obs of the new last step = the observation of the dropped one (stored by the policy warps)
#pragma unroll
                    for (int f = 0; f < 5; ++f)
                        if (f < F) a.next_obs[((uint64_t)(len - 1) * F + f) * a.E + e] = __ldcg(a.obs + ((uint64_t)len * F + f) * a.E + e);
                    eps += 1.0;
                }
            }
            a.lane_len[e] = len;
            a.lane_flags[e] = (uint8_t)flags;
            st.v[ST_STORED_STEPS] = (double)len;
            st.v[ST_STORED_EPS] = eps;
            contributes = true;
        }
    }
    __shared__ double red[32][ST_COUNT];
    block_reduce_stats(st, contributes, red, a.partials);
}
