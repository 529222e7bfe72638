// rollout_ws6.cuh -- K2q: the warp-specialised CartPole rollout (RL_LANES_WARP_SPECIALIZED at any size, `lanes_per_env = 0`
// for the categorical actor on Philox noise up to 64 envs per SM).  Included by rollout.cu inside its anonymous namespace.
//
// K2c<8> (rollout.cu) has each warp carry 4 envs x 8 threads and issue BOTH halves of the step chain: the policy
// (obs -> hidden layer -> logit difference -> compare) and the f64 dynamics, the latter redundantly in all 8 threads of an
// env.  K2q splits the chain by warp.  A CTA owns 4 x policy_warps envs (1 .. 8 policy warps, launch_ws6's shape rule) and
// has twelve warps:
//  * the POLICY warps, 4 envs x 8 threads each, with exactly K2c<8>'s register-resident hidden layer;
//  * one DYNAMICS warp, lane = env, which evaluates the step for BOTH actions in the same thread (four independent chains:
//    2 actions x 2 friction signs; everything that does not depend on the action -- sin / cos, the reciprocals, beta -- is
//    computed once), so the select after the action needs no shuffles;
//  * one AUX warp that draws every Philox block: the actor's uniform of each step, as its logit-space threshold, and the
//    would-be reset state of each step.  It fills them WS_CHUNK steps at a time into WS_RING-step shared-memory rings, up
//    to WS_AHEAD steps ahead of the dynamics warp.  Progress is three counters in shared memory, not a barrier: `prod`
//    (steps filled, written by the aux warp), `cons` (the dynamics warp's iteration, posted every fourth) and `done` (the
//    dynamics loop is over);
//  * warps without a role (QK_ROLE_IDLE), which wait at the final barrier.
// Warp w runs on sub-partition w % 4, and the dynamics warp has its sub-partition's scheduler to itself: per-phase clocks
// (scripts/ws_clocks.sh, profiles/r2_summary.md section 5) put the step cycle on the dynamics warp's own instruction
// stream, ~75 % issue-busy, and a dynamics stream that shared its scheduler with policy warps took ~1150 clk per step
// instead of ~850.  Further work therefore leaves the dynamics warp: the step record's successor code and reward are
// stored one iteration later by two idle threads of the env's policy group (the row carries the previous step's code),
// episode statistics are integer counters, and finalize_last_episode reads the dropped observation back from the
// trajectory.
// No work around the launch: the dynamics lanes fill `succ` with RL_PAD past their last step, and the last CTA to finish
// sums every CTA's statistics (finalize_stat: rollout_finalize_kernel's sum, in its order).
// The hand-off has one row per env: dynamics publishes the row of step i -> barrier 1 -> policy samples -> action ->
// barrier 2 -> dynamics selects.  The grid is one CTA per 4 x policy_warps envs, so any number of waves runs.  Same
// operations on the same operands as K2c<8> (summation order of the logits included): bit-identical trajectories and
// summaries (tests/test_gpu_envs.py).  Philox noise and the categorical actor only.
// The earlier six-warp, 16-env kernel for up to 16 envs per SM was measured against K2q and retired
// (profiles/r2_summary.md section 5, profiles/r4_k2q_small_e.md, git history).
#pragma once

constexpr int WS_RING = 16, WS_CHUNK = 4, WS_AHEAD = 11;  // the aux warp's rings

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

constexpr int QK_ENVS = 32, QK_THREADS = 384, QK_POLICY_WARPS = 8;  // at most; RolloutArgs::policy_warps x 4 envs are used
constexpr int QK_ROLE_DYN = 8, QK_ROLE_AUX = 9, QK_ROLE_IDLE = 15;

struct QkShared {
    float4 sw4[4 * GK_PAIRS];
    float tail[4 + GK_REM_TABLE_MAX];
    // rows[env]: (x, x', theta, theta') | (remaining, flags, -, -); flags: bit 0 this env takes the step, bit 1 some env of
    // the CTA does, bit 2 the env took the previous step, bits 8.. that step's successor code
    float4 rows[QK_ENVS][2];
    uint32_t act[QK_ENVS];
    float thr[WS_RING][QK_ENVS];       // logit-space thresholds
    double2 slot[WS_RING][QK_ENVS][2]; // would-be reset states (x, x') | (theta, theta')
    uint32_t prod, cons, done, last;
};
#define QK_OFF(member) ((uint32_t)offsetof(QkShared, member))
constexpr uint32_t QK_ACTIVE = 1u, QK_ANY = 2u, QK_PREV_ACTIVE = 4u;

__global__ void __launch_bounds__(QK_THREADS, 1) rollout_cartpole_ws6_kernel(CartPoleEnv::Params p, RolloutArgs a) {
    using EnvT = CartPoleEnv;
    constexpr int LANES = 8, PPL = GK_PAIRS / LANES;
    constexpr unsigned FULL = 0xffffffffu;
    extern __shared__ __align__(16) unsigned char gk_smem[];
    QkShared &sh = *reinterpret_cast<QkShared *>(gk_smem);
    // (through a shuffle: ptxas otherwise rematerialises the window base at its uses in the loops)
    const uint32_t sb = __shfl_sync(FULL, (uint32_t)__cvta_generic_to_shared(gk_smem), 0);
    const bool rem_table = p.max_steps != 0 && p.max_steps < GK_REM_TABLE_MAX;
    stage_pair_weights(a.net, sh.sw4, sh.tail, p, rem_table ? (int)p.max_steps + 1 : 0);
    const uint32_t rem_addr = sb + QK_OFF(tail) + 8;
    auto remaining_feature = [&](uint32_t r) {
        return p.max_steps == 0 ? 0.0f : rem_table ? smem_ldf(rem_addr + 4u * r) : (float)__ddiv_rn((double)r, (double)p.max_steps);
    };
    const int hw_warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // roles by hardware warp (warp w runs on sub-partition w % 4)
    const int warp = (int)((a.role_table >> (4 * hw_warp)) & 15u);  // policy warp index, or one of the role codes
    const bool is_dyn = warp == QK_ROLE_DYN, is_aux = warp == QK_ROLE_AUX, is_idle = warp == QK_ROLE_IDLE;
    const int cta_envs = 4 * a.policy_warps, QK_SYNC = 32 * (a.policy_warps + 1);
    const uint64_t e_base = (uint64_t)blockIdx.x * (uint64_t)cta_envs;
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

    // ---- aux: one chunk = WS_CHUNK steps x 32 envs; lane = env ----
    const RlPhiloxKeys keys = rl_philox_keys(seed);
    auto aux_fill = [&](uint32_t k0) {
        const int el = lane;
        const uint64_t eg = e_base + el, lg = a.lane_offset + (eg < a.E ? eg : 0);  // (lanes past the CTA's envs: unused slots)
#pragma unroll 1
        for (int j = 0; j < WS_CHUNK; ++j) {
            const uint32_t k = k0 + (uint32_t)j;
            const uint32_t ring = k & (WS_RING - 1);
            uint32_t oa[4], o0[4], o1[4];
            // policies/actor.rs:42-55: the actor's uniform of step k as the logit-space threshold (rl_logit_threshold)
            rl_philox4x32_10_keyed((uint32_t)lg, (uint32_t)(lg >> 32), t0 + k, (uint32_t)RL_STREAM_ACTOR * 64u, keys, oa);
            // cartpole.rs:103-115: four uniform draws in field order = blocks 0 (x, x') and 1 (theta, theta')
            rl_philox4x32_10_keyed((uint32_t)lg, (uint32_t)(lg >> 32), t0 + k, (uint32_t)RL_STREAM_ENV_RESET * 64u, keys, o0);
            rl_philox4x32_10_keyed((uint32_t)lg, (uint32_t)(lg >> 32), t0 + k, (uint32_t)RL_STREAM_ENV_RESET * 64u + 1u, keys, o1);
            smem_stf(sb + QK_OFF(thr) + 4u * (ring * QK_ENVS + el), rl_logit_threshold_fast(rl_u32_to_f32(oa[0])));
            const double x = rl_u64_to_uniform((uint64_t)o0[0] | ((uint64_t)o0[1] << 32), p.reset_low, p.reset_scale);
            const double xd = rl_u64_to_uniform((uint64_t)o0[2] | ((uint64_t)o0[3] << 32), p.reset_low, p.reset_scale);
            const double th = rl_u64_to_uniform((uint64_t)o1[0] | ((uint64_t)o1[1] << 32), p.reset_low, p.reset_scale);
            const double thd = rl_u64_to_uniform((uint64_t)o1[2] | ((uint64_t)o1[3] << 32), p.reset_low, p.reset_scale);
            const uint32_t sa = sb + QK_OFF(slot) + 32u * (ring * QK_ENVS + el);
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
    if (is_aux && lane == 0) smem_stu(sb + QK_OFF(prod), 2 * WS_CHUNK);

    if (is_idle) {
        // (keeps the dynamics warp's scheduler free; waits at the barrier below)
    } else if (is_aux) {
        // ------------------------------ aux warp ------------------------------
        uint32_t k0 = 2 * WS_CHUNK;
        while (k0 <= cap + 1) {
            // slots of steps k0 - 16 .. k0 - 13 are reused: their readers (thresholds at iteration k, reset states at
            // k - 1) are done once the dynamics warp is at iteration >= k0 - 12
            uint32_t c = smem_ldu(sb + QK_OFF(cons));
            bool over = false;
            while (k0 > c + WS_AHEAD) {
                if (smem_ldu(sb + QK_OFF(done))) { over = true; break; }
                __nanosleep(64);
                c = smem_ldu(sb + QK_OFF(cons));
            }
            if (over) break;
            aux_fill(k0);
            __threadfence_block();
            __syncwarp();
            k0 += WS_CHUNK;
            if (lane == 0) smem_stu(sb + QK_OFF(prod), k0);
        }
    } else if (is_dyn) {
        // ------------------------------ dynamics warp: lane = env ------------------------------
        const int el = lane;
        const uint64_t e = e_base + el;
        const bool valid = el < cta_envs && e < a.E;
        const uint64_t e_safe = valid ? e : 0;
        const float rem_full = remaining_feature(p.max_steps);
        const uint32_t slot0 = sb + QK_OFF(slot) + 32u * (uint32_t)el, row = sb + QK_OFF(rows) + 32u * (uint32_t)el;
        const uint32_t act_addr = sb + QK_OFF(act) + 4u * (uint32_t)el;
        // the reset state of noise step t0 + k, from the ring the aux warp keeps ahead
        auto fresh_state = [&](uint32_t k, EnvT::State &f) {
            const uint32_t sa = slot0 + 32u * QK_ENVS * (k & (WS_RING - 1));
            const double2 lo = smem_ldd2(sa), hi = smem_ldd2(sa + 16);
            f.x = lo.x; f.xd = lo.y; f.th = hi.x; f.thd = hi.y;
            f.meta = 0x80000000u | p.max_steps;
        };
        // step_fast's parameters and coefficients in registers for the whole loop.  Left to ptxas, they are reloaded from
        // the constant bank on every step, about twenty loads on the dynamics warp's stream, which is what bounds the
        // step cycle; ptxas does not rematerialise a shuffle's result.
        EnvT::Params q = p;
        for (double *v : {&q.gravity, &q.mass_pole, &q.length_half_pole, &q.friction_cart, &q.friction_pole, &q.time_step,
                          &q.action_force, &q.max_pos, &q.max_angle, &q.total_weight, &q.inv_total_mass, &q.mass_length_pole})
            *v = __shfl_sync(FULL, *v, 0);
        double coef[14];
#pragma unroll
        for (int c = 0; c < 14; ++c) coef[c] = __shfl_sync(FULL, rl_cartpole_sincos_coef[c], 0);
        // beta's divisor is the constant mass_length_pole: its reciprocal (MUFU.RCP64H and the Newton steps, which ptxas left
        // inside the loop) once, and the slack bound of the step loop, which it otherwise reloads from the constant bank
        const double rcp_ml = __shfl_sync(FULL, EnvT::rcp_fast(q.mass_length_pole), 0);
        const uint32_t slack = __shfl_sync(FULL, a.slack, 0);
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
        bool any = __any_sync(FULL, n > 0);
        smem_st4(row, make_float4((float)s.x, (float)s.xd, (float)s.th, (float)s.thd));
        smem_st4(row + 16, make_float4(obs4, __uint_as_float((n > 0 ? QK_ACTIVE : 0u) | (any ? QK_ANY : 0u)), 0.0f, 0.0f));
        __syncwarp();
        named_bar_arrive(1, QK_SYNC);
        uint32_t it = 0;                                  // loop counter (= step index of the envs still active)
        uint32_t i = 0, cur_len = 0, n_eps = 0;           // steps stored, length of the running episode, episodes ended
        unsigned long long sum_el = 0ull, sum_el2 = 0ull; // sum of episode lengths and of their squares
        int succ_last = RL_TERMINATE, succ_prev = RL_TERMINATE;
#ifdef RL_WS_CLOCKS
        long long ck[5] = {0, 0, 0, 0, 0};
#endif
        while (any) {
            WS_CLK(c0, s.x, it);
            const bool active = n > 0;
            if ((it & 3u) == 0u && lane == 0) smem_stu(sb + QK_OFF(cons), it);
            if ((it & 3u) == 3u) {  // the reset states of steps it + 1 .. it + 4
                while (smem_ldu(sb + QK_OFF(prod)) < it + 5u) { }
                asm volatile("fence.acq_rel.cta;" ::: "memory");
            }
            // before the action is known: the step for both actions, the would-be reset state, and the `remaining` feature
            // of the next observation
            EnvT::State c0s = s, c1s = s;
            // (a state that terminates is replaced by `fresh` below: step_fast need not keep it)
            const int sc0 = EnvT::step_fast<false>(q, c0s, 0u, coef, rcp_ml);
            const int sc1 = EnvT::step_fast<false>(q, c1s, 1u, coef, rcp_ml);
            EnvT::State fresh;
            fresh_state(it + 1, fresh);
            const uint32_t r_now = s.meta & 0x7FFFFFFFu;
            const float rem_cont = remaining_feature(r_now > 0 ? r_now - 1 : 0);
            WS_CLK(c1, c0s.x + c1s.x + c0s.thd + c1s.thd + fresh.x, (uint32_t)(sc0 + sc1) + __float_as_uint(rem_cont));
            named_bar_sync(2, QK_SYNC);
            WS_CLK(c2, 0.0, 0u);
            const bool one = smem_ldu(act_addr) != 0u;
            EnvT::State post;
            post.x = one ? c1s.x : c0s.x; post.xd = one ? c1s.xd : c0s.xd;
            post.th = one ? c1s.th : c0s.th; post.thd = one ? c1s.thd : c0s.thd;
            post.meta = one ? c1s.meta : c0s.meta;
            const int sc = one ? sc1 : sc0;
            const bool ended = sc != RL_CONTINUE;  // steps.rs:116-124: the next call starts a new episode
            s.x = ended ? fresh.x : post.x; s.xd = ended ? fresh.xd : post.xd;
            s.th = ended ? fresh.th : post.th; s.thd = ended ? fresh.thd : post.thd;
            s.meta = ended ? fresh.meta : post.meta;
            uint32_t n_next = n;
            if (active) {
                n_next = n - 1;
                if (ended && n_next <= slack) n_next = 0;  // take_steps.rs:83-88
            }
            const bool any_next = __any_sync(FULL, n_next > 0);
            smem_st4(row, make_float4((float)s.x, (float)s.xd, (float)s.th, (float)s.thd));
            smem_st4(row + 16, make_float4(ended ? rem_full : rem_cont,
                                         __uint_as_float((n_next > 0 ? QK_ACTIVE : 0u) | (any_next ? QK_ANY : 0u) |
                                                         (active ? QK_PREV_ACTIVE : 0u) | ((uint32_t)sc << 8)),
                                         0.0f, 0.0f));
            __syncwarp();
            named_bar_arrive(1, QK_SYNC);
            WS_CLK(c3, 0.0, 0u);
            // ---- off the chain ----
            if (active && sc == RL_INTERRUPT) {  // rare: once per max_steps; the post-step observation (remaining == 0)
                const uint64_t io = (uint64_t)i * FE + e_safe;
                a.next_obs[io] = (float)post.x;
                a.next_obs[io + a.E] = (float)post.xd;
                a.next_obs[io + 2 * a.E] = (float)post.th;
                a.next_obs[io + 3 * a.E] = (float)post.thd;
                if (F > 4) a.next_obs[io + 4 * a.E] = remaining_feature(post.meta & 0x7FFFFFFFu);
            }
            // episode statistics (summary.rs:198-216) as exact integer counters
            const bool ep_end = active && ended;
            i += active ? 1u : 0u;
            cur_len += active ? 1u : 0u;
            n_eps += ep_end ? 1u : 0u;
            sum_el += ep_end ? (unsigned long long)cur_len : 0ull;
            sum_el2 += ep_end ? (unsigned long long)cur_len * cur_len : 0ull;
            cur_len = ep_end ? 0u : cur_len;
            succ_prev = active ? succ_last : succ_prev;
            succ_last = active ? sc : succ_last;
            n = n_next;
            any = any_next;
            it += 1;
#ifdef RL_WS_CLOCKS
            const long long c4 = ws_clk((double)sum_el2, i + cur_len);
            ck[0] += c1 - c0; ck[1] += c2 - c1; ck[2] += c3 - c2; ck[3] += c4 - c3; ck[4] += 1;
#endif
        }
#ifdef RL_WS_CLOCKS
        if (lane == 0 && ck[4] > 0 && (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1))
            printf("K2q dyn cta %d: %lld iterations; clk per iteration: step for both actions %.1f, wait for the action %.1f, "
                   "select + publish %.1f, bookkeeping %.1f\n", (int)blockIdx.x, ck[4], (double)ck[0] / ck[4], (double)ck[1] / ck[4],
                   (double)ck[2] / ck[4], (double)ck[3] / ck[4]);
#endif
        if (lane == 0) smem_stu(sb + QK_OFF(done), 1u);
        // (kept for after the barrier that ends the loops)
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
        // Thread `sub` stores ONE column of the step records, one pointer and one stride each: sub < F (<= 5) observation
        // feature sub of this step, sub == 5 its action and -- one iteration later, the row carries the previous step's code --
        // sub == 6 the successor code, sub == 7 the reward (their pointers start one row behind).
        const bool lagged = sub >= 6, is_word = sub != 5 && sub != 6;
        const bool has_column = valid && (sub >= 5 || sub < F);
        uint8_t *col_ptr = sub < 5    ? reinterpret_cast<uint8_t *>(a.obs + (uint64_t)sub * a.E + e_safe)
                           : sub == 5 ? a.action + e_safe
                           : sub == 6 ? a.succ + e_safe - a.E
                                      : reinterpret_cast<uint8_t *>(a.reward + e_safe - a.E);
        const uint64_t col_stride = sub < 5 ? 4ull * FE : sub == 7 ? 4ull * a.E : a.E;
        const uint32_t col_flag = lagged ? QK_PREV_ACTIVE : QK_ACTIVE;
        const uint32_t row = sb + QK_OFF(rows) + 32u * (uint32_t)el, mine_addr = row + 4u * (uint32_t)(sub < 5 ? sub : 0);
        const uint32_t thr_addr = sb + QK_OFF(thr) + 4u * (uint32_t)el, act_addr = sb + QK_OFF(act) + 4u * (uint32_t)el;
#ifdef RL_WS_CLOCKS
        long long pk[4] = {0, 0, 0, 0};
#endif
        for (uint32_t i = 0;; ++i) {
            WS_CLK(q0, 0.0, i);
            // (No poll of `prod` here: the dynamics warp saw the thresholds of steps <= i + 1 published before it arrived
            // at barrier 1 for the row of step i -- it polls every fourth iteration, up to four steps ahead -- and the
            // barrier orders that observation before the load below.)
            named_bar_sync(1, QK_SYNC);
            WS_CLK(q1, 0.0, 0u);
            const float4 ov = smem_ld4(row);
            const float4 tv = smem_ld4(row + 16);
            const float mine = smem_ldf(mine_addr);
            const float theta = smem_ldf(thr_addr + 4u * QK_ENVS * (i & (WS_RING - 1)));
            const float ob4 = tv.x;
            const uint32_t flags = __float_as_uint(tv.y);
            // this thread's column of the step record (sub >= 6: of the previous step); off the chain except at the end
            auto store_column = [&](uint32_t action_now) {
                if (has_column && (flags & col_flag) != 0u) {
                    if (is_word) *reinterpret_cast<float *>(col_ptr) = lagged ? 1.0f : mine;  // reward: cartpole.rs:140
                    else *col_ptr = (uint8_t)(lagged ? flags >> 8 : action_now);
                }
            };
#ifdef RL_WS_CLOCKS
            if ((flags & QK_ANY) == 0u && warp == 0 && lane == 0 && pk[3] > 0 && (blockIdx.x == 0 || blockIdx.x == gridDim.x - 1))
                printf("K2q policy cta %d: %lld iterations; clk per iteration: wait for the row %.1f, row -> action published %.1f, "
                       "record stores %.1f\n", (int)blockIdx.x, pk[3], (double)pk[0] / pk[3], (double)pk[1] / pk[3], (double)pk[2] / pk[3]);
#endif
            if ((flags & QK_ANY) == 0u) {
                if (lagged) store_column(0u);
                break;
            }
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
            if (sub == 0) smem_stu(act_addr, action);
            __syncwarp();
            named_bar_arrive(2, QK_SYNC);
            WS_CLK(q2, 0.0, action);
            // ---- off the chain: the step record ----
            store_column(action);
            col_ptr += col_stride;
#ifdef RL_WS_CLOCKS
            const long long q3 = ws_clk(0.0, (uint32_t)(uintptr_t)col_ptr);
            pk[0] += q1 - q0; pk[1] += q2 - q1; pk[2] += q3 - q2; pk[3] += 1;
#endif
        }
    }
    __syncthreads();  // the policy warps' stores of the step records are visible to the dynamics warp from here on
    if (is_dyn) {
        const uint64_t e = e_base + lane;
        if (lane < cta_envs && e < a.E) {
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
            // the slots no step was stored in (rl_rollout fills `succ` with RL_PAD before the other kernels)
            for (uint64_t k = i; k < a.Tcap; ++k) a.succ[k * a.E + e] = RL_PAD;
            a.lane_len[e] = len;
            a.lane_flags[e] = (uint8_t)flags;
            st.v[ST_STORED_STEPS] = (double)len;
            st.v[ST_STORED_EPS] = eps;
            contributes = true;
        }
    }
    __shared__ double red[32][ST_COUNT];
    block_reduce_stats(st, contributes, red, a.partials);
    // The last CTA to finish publishes the totals (each CTA's partials are visible device-wide before it takes its
    // ticket; that CTA puts the ticket back to 0 for the next launch).
    if (threadIdx.x < ST_COUNT) __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) sh.last = atomicAdd(a.ticket, 1u) == gridDim.x - 1 ? 1u : 0u;
    __syncthreads();
    if (sh.last) {
        if (hw_warp < ST_COUNT)
            finalize_stat(a.partials, (int)gridDim.x, hw_warp, lane, a.partials - ST_COUNT, a.traj_counts, a.summary_host);
        if (threadIdx.x == 0) *a.ticket = 0u;
    }
}
