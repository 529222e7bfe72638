// gru_step_tc.cuh -- K8s: the fused rollout with the rl2-sized recurrent policy (Chain<Gru(F -> 128), Linear(128 -> A)>) as TWO
// launches per step over all envs of the GPU: the GRU cell on the tensor cores (gru_big_tc.cuh: [E x (F + 128)] . [(F + 128) x
// 512] as bf16-piece tcgen05 MMAs, lanes on the TMEM lanes, gates in the TMEM epilogue) and an "owner" kernel, one thread per
// env, that folds relu(h') into the logits, samples, steps the env, stores the step record and writes the next
// observation.  K8h (gru_tile.cuh) keeps everything of a 64-env tile inside one persistent CTA but runs the cell as an FP32
// FFMA2 GEMM (56 % of the FMA roof, 338 M env-steps/s); here the cell costs ~10 us per step for 18 944 envs and the env
// state lives in a global array between launches.  Included by gru.cu after gru_tile.cuh (GtOwner, SeqArgs, steps.cuh).
#pragma once

template <class EnvT, bool REPLAY>
__global__ void __launch_bounds__(128) seq_owner_init_kernel(typename EnvT::Params p, SeqArgs a, GtOwner<EnvT, REPLAY> *owners,
                                                            float *__restrict__ xplane, float *__restrict__ hplane) {
    constexpr int MF = EnvT::MAXF;
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= a.E) return;
    GtOwner<EnvT, REPLAY> o;
    o.st.init();
    o.i = 0;
    o.succ_last = o.succ_prev = RL_TERMINATE;
    o.n = a.min_steps ? a.min_steps + a.slack : 0;  // take_steps.rs:20-31
#pragma unroll
    for (int f = 0; f < MF; ++f) o.last_obs[f] = 0.0f;
    o.nz.init(a.noise, a.lane_offset + e, e);
    float obs[MF];
#pragma unroll
    for (int f = 0; f < MF; ++f) obs[f] = 0.0f;
    if (o.n > 0) {  // train.rs:135: every period starts fresh episodes
        o.nz.set_step(a.noise.step_counter);
        EnvT::template reset<REPLAY>(p, o.s, o.nz);
        EnvT::observe(p, o.s, obs);
    }
#pragma unroll
    for (int f = 0; f < MF; ++f)
        if (f < a.F) xplane[(uint64_t)f * a.E + e] = obs[f];
    for (int j = 0; j < GT_H; ++j) hplane[(uint64_t)j * a.E + e] = 0.0f;  // SeqIterative::initial_state (gru.rs:23-28)
    owners[e] = o;
}

// One step of every env that still collects: logits from h' (hnew plane), sample, record, env step, next observation.
// (Two CTAs per SM: at 157 registers only one fitted and the 296 CTAs of 18 944 envs ran as two waves -- 10.28 -> 8.66 ms
// per 199-step rollout.  A unit-major weight layout read with LDS.128 was measured slower: 9.12 ms.)
template <class EnvT, bool REPLAY>
__global__ void __launch_bounds__(256, 2) seq_owner_step_kernel(typename EnvT::Params p, SeqArgs a, GtOwner<EnvT, REPLAY> *owners,
                                                            float *__restrict__ xplane, float *__restrict__ hnew) {
    constexpr int MF = EnvT::MAXF, MA = EnvT::MAXA;
    extern __shared__ float osm[];  // lin_w [A][128], lin_b [A]
    const int F = a.F, A = a.A;
    {
        const float *lw = a.net.params + (size_t)3 * GT_H * F + (size_t)3 * GT_H * GT_H + 6 * GT_H;
        for (int i = threadIdx.x; i < A * GT_H + A; i += blockDim.x) osm[i] = lw[i];
    }
    __syncthreads();
    // four threads per env (K8h's arrangement): thread (env, part) folds units part, part + 4, ... into the logits, two
    // shuffles add the parts, part 0 owns the env.  (One thread per env left one warp per scheduler: 46 us per step.)
    const uint64_t gt = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, E = a.E;
    const uint64_t e = gt >> 2;
    const int part = (int)(gt & 3);
    const bool valid = e < E;
    const uint64_t e_safe = valid ? e : 0;
    const bool live = valid && owners[e_safe].n > 0;
    float zl[MA];
#pragma unroll
    for (int k = 0; k < MA; ++k) zl[k] = 0.0f;
    {
        float hv[GT_H / 4];
#pragma unroll
        for (int jj = 0; jj < GT_H / 4; ++jj) hv[jj] = live ? hnew[(uint64_t)(part + 4 * jj) * E + e_safe] : 0.0f;
#pragma unroll
        for (int jj = 0; jj < GT_H / 4; ++jj) {
            const float av = rl_activate(a.net.act, hv[jj]);
#pragma unroll
            for (int k = 0; k < MA; ++k)
                if (k < A) zl[k] = fmaf(osm[k * GT_H + part + 4 * jj], av, zl[k]);
        }
    }
#pragma unroll
    for (int k = 0; k < MA; ++k) {
        zl[k] += __shfl_xor_sync(0xffffffffu, zl[k], 1);
        zl[k] += __shfl_xor_sync(0xffffffffu, zl[k], 2);
        zl[k] += k < A ? osm[A * GT_H + k] : 0.0f;
    }
    if (!live || part != 0) return;
    GtOwner<EnvT, REPLAY> &og = owners[e];
    GtOwner<EnvT, REPLAY> o = og;
    const uint32_t t0 = a.noise.step_counter, i = o.i;
    o.nz.set_step(t0 + i);
    const float u = rl_u32_to_f32(o.nz.template next_u32<RL_STREAM_ACTOR>());
    const uint32_t action = categorical_sample<MA>(zl, A, u);
    {  // the step's observation: loads first, stores after (written pairwise the loads queued behind the stores)
        const float *__restrict__ xin = xplane;
        float *__restrict__ obs_out = a.obs;
        float xv[MF];
#pragma unroll
        for (int f = 0; f < MF; ++f) xv[f] = f < F ? xin[(uint64_t)f * E + e] : 0.0f;
#pragma unroll
        for (int f = 0; f < MF; ++f)
            if (f < F) {
                obs_out[((uint64_t)i * F + f) * E + e] = xv[f];
                o.last_obs[f] = xv[f];
            }
    }
    float r;
    const int sc = EnvT::template step<REPLAY>(p, o.s, action, o.nz, r);
    float obs[MF];
    if (sc == RL_INTERRUPT) {
        EnvT::observe(p, o.s, obs);
#pragma unroll
        for (int f = 0; f < MF; ++f)
            if (f < F) a.next_obs[((uint64_t)i * F + f) * E + e] = obs[f];
    }
    if (sc != RL_CONTINUE) {
        o.nz.set_step(t0 + i + 1);
        EnvT::template reset<REPLAY>(p, o.s, o.nz);
        for (int j = 0; j < GT_H; ++j) hnew[(uint64_t)j * E + e] = 0.0f;  // steps.rs:116-124: actor.initial_state
    }
    EnvT::observe(p, o.s, obs);
#pragma unroll
    for (int f = 0; f < MF; ++f)
        if (f < F) xplane[(uint64_t)f * E + e] = obs[f];
    a.action[(uint64_t)i * E + e] = (uint8_t)action;
    a.reward[(uint64_t)i * E + e] = r;
    a.succ[(uint64_t)i * E + e] = (uint8_t)sc;
    o.st.push(r, sc);
    o.succ_prev = o.succ_last;
    o.succ_last = sc;
    o.i = i + 1;
    uint32_t n = o.n - 1;
    if (sc != RL_CONTINUE && n <= a.slack) n = 0;  // take_steps.rs:83-88
    o.n = n;
    og = o;
}

// VecBuffer::end_experience -> finalize_last_episode (buffers/mod.rs:237-261) and the block partials of the summary sums
template <class EnvT, bool REPLAY>
__global__ void __launch_bounds__(128) seq_owner_finish_kernel(SeqArgs a, GtOwner<EnvT, REPLAY> *owners) {
    constexpr int MF = EnvT::MAXF;
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int F = a.F;
    LaneStats st;
    st.init();
    if (e < a.E) {
        GtOwner<EnvT, REPLAY> &o = owners[e];
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
    __shared__ double red[4][ST_COUNT];
    block_reduce_stats(st, e < a.E, red, a.partials);
}

template <class EnvT, bool REPLAY>
rl_status launch_seq_stepped_t(rl_ctx *ctx, const typename EnvT::Params &p, SeqArgs &a, char *scratch) {
    using Owner = GtOwner<EnvT, REPLAY>;
    const int F = a.F, A = a.A;
    const uint64_t E = a.E;
    auto al = [](size_t b) { return (b + 255) / 256 * 256; };
    char *q = scratch;
    void *prepared = q; q += rl_seq_big_prepared_bytes(F, GT_H);
    Owner *owners = reinterpret_cast<Owner *>(q); q += al(E * sizeof(Owner));
    float *xplane = reinterpret_cast<float *>(q); q += al((size_t)F * E * 4);
    float *hA = reinterpret_cast<float *>(q); q += al((size_t)GT_H * E * 4);
    float *hB = reinterpret_cast<float *>(q);
    const unsigned grid = rl_grid_for(E, 128);
    const size_t osmem = (size_t)(A * GT_H + A) * sizeof(float);
    RL_TRY(rl_seq_big_prepare(ctx, a.net.params, F, GT_H, prepared));
    RL_LAUNCH(ctx, (seq_owner_init_kernel<EnvT, REPLAY>), grid, 128, 0, p, a, owners, xplane, hA);
    const uint32_t cap = a.min_steps ? a.min_steps + a.slack : 0;  // no env takes more steps than this
    float *hcur = hA, *hnxt = hB;
    for (uint32_t t = 0; t < cap; ++t) {
        RL_TRY(rl_seq_big_cell(ctx, prepared, F, GT_H, xplane, hcur, E, hnxt));
        RL_LAUNCH(ctx, (seq_owner_step_kernel<EnvT, REPLAY>), rl_grid_for(4 * E, 256), 256, osmem, p, a, owners, xplane, hnxt);
        float *tmp = hcur; hcur = hnxt; hnxt = tmp;
    }
    RL_LAUNCH(ctx, (seq_owner_finish_kernel<EnvT, REPLAY>), grid, 128, 0, a, owners);
    return RL_OK;
}

template <class EnvT>
size_t seq_stepped_scratch_bytes(int F, uint64_t E) {
    auto al = [](size_t b) { return (b + 255) / 256 * 256; };
    const size_t own = sizeof(GtOwner<EnvT, true>) > sizeof(GtOwner<EnvT, false>) ? sizeof(GtOwner<EnvT, true>) : sizeof(GtOwner<EnvT, false>);
    return rl_seq_big_prepared_bytes(F, GT_H) + al(E * own) + al((size_t)F * E * 4) + 2 * al((size_t)GT_H * E * 4) + 256;
}

template <class EnvT>
rl_status launch_seq_stepped(rl_ctx *ctx, const typename EnvT::Params &p, SeqArgs &a, bool replay) {
    char *scratch;
    RL_TRY(rl_ctx_scratch2(ctx, seq_stepped_scratch_bytes<EnvT>(a.F, a.E), (void **)&scratch));
    if (replay) return launch_seq_stepped_t<EnvT, true>(ctx, p, a, scratch);
    return launch_seq_stepped_t<EnvT, false>(ctx, p, a, scratch);
}
