// gru.cu -- Chain<Gru, Linear> policy module and its fused rollout (BASELINE config 4: bandit meta-env with a
// GRU policy).
//
// Reference: Gru / RnnBase (src/torch/modules/seq/rnn/gru.rs:23-102, rnn/mod.rs:166-280), Chain
// (src/torch/modules/chain.rs:12-186), Linear (ff/linear.rs:108-123), PolicyActor::act
// (src/torch/agents/policies/actor.rs:42-55), Steps::step (src/simulation/steps.rs:113-168: the actor's
// episode state -- the GRU hidden state -- is re-initialised to zeros whenever a new episode starts).
//
// libtorch's gru_cell (what Tensor::gru_cell and gru_data evaluate per step), gate order r, z, n:
//   r = sigmoid(W_ir x + b_ir + W_hr h + b_hr)      z = sigmoid(W_iz x + b_iz + W_hz h + b_hz)
//   n = tanh(W_in x + b_in + r * (W_hn h + b_hn))   h' = (h - n) * z + n
//
// The same kernels run DqnActor::act (dqn.rs:360-379) for a recurrent Q-network (SeqArgs::eps_greedy): epsilon-greedy on the
// module's outputs, the hidden state held where the actor explores.
//
//  K8a rollout_seq_kernel<EnvT, HMAX>   one thread per env; hidden state in registers (hidden <= 8) or
//                                       thread-local memory (hidden <= 128); weights read as warp-wide
//                                       broadcasts from shared memory when they fit, else through L1.
//  K8b grunet_seq_kernel<HMAX>          SeqPacked::seq_packed over a stored trajectory (one thread per lane).
//
//  K8h rollout_seq_tile_kernel         gru_tile.cuh: hidden 128 (the rl2-sized module) as a register-tiled FP32 GEMM
//                                       per step over 64-env CTAs, weights streamed through shared memory.
//
// For the benches/rnn.rs-sized module (hidden 4) the per-step cost is ~150 FMAs and the kernel is bound by the
// trajectory write stream and the env arithmetic, like K2a.  The rl2-sized module (hidden 128, 1.1e5 FLOP per
// env-step) is a dense [E, F+H] x [F+H, 3H] GEMM per step: K8h runs it at 56 % of the FP32 FMA roof (27x K8a);
// K8a stays as the cross-check (RL_GRU_KERNEL=thread) and for hidden sizes between 9 and 127.
#include <cstdlib>
#include <cstring>
#include <type_traits>

#include "handles.cuh"
#include "tcgen05.cuh"
#include "steps.cuh"

struct rl_grunet {
    rl_ctx *ctx = nullptr;
    int in_dim = 0, hidden = 0, out_dim = 0;
    rl_activation act = RL_ACT_RELU;
    int cell = RL_CELL_GRU;
    uint64_t n_params = 0;
    float *params = nullptr;  // w_ih[G H,in], w_hh[G H,H], b_ih[G H], b_hh[G H], kernel[out,H], bias[out]; G = 3 (GRU) or 4 (LSTM)
    float *wt = nullptr;      // K8h: k-major copy of w_ih / w_hh, [in + H][3H] (rebuilt before every tiled rollout)
};

namespace {

struct GruView {
    const float *params;
    int F, H, A, act;
    int cell;
    __host__ __device__ uint64_t count() const {
        const uint64_t G = rl_cell_gates(cell);
        return G * H * F + G * H * H + 2 * G * H + (uint64_t)A * H + A;
    }
};

__device__ __forceinline__ float sigmoidf_ref(float v) { return 1.0f / (1.0f + expf(-v)); }

// One gru_cell + activation + Linear for this thread's env.  `w` points at the parameters (shared or global).
// EXACT: the sizes ARE (MAXF, HMAX, MAXA) -- no padded iterations, no predicates (BASELINE config 4: 6 / 4 / 2).
template <int HMAX, int MAXF, int MAXA, bool EXACT = false>
__device__ __forceinline__ void grunet_step(const GruView &m, const float *__restrict__ w, const float *x, float *h, float *z) {
    const int F = EXACT ? MAXF : m.F, H = EXACT ? HMAX : m.H, A = EXACT ? MAXA : m.A;
    const float *w_ih = w, *w_hh = w_ih + (size_t)3 * H * F, *b_ih = w_hh + (size_t)3 * H * H, *b_hh = b_ih + 3 * H;
    const float *lin_w = b_hh + 3 * H, *lin_b = lin_w + (size_t)A * H;
    // HMAX <= 8: everything unrolled, hidden state in registers.  Larger: plain loops over thread-local arrays.
    constexpr bool SMALL = HMAX <= 8;
    float hn[HMAX];
#pragma unroll(SMALL ? HMAX : 1)
    for (int j = 0; j < (SMALL ? HMAX : H); ++j) {
        if (SMALL && j >= H) break;
        float gi[3], gh[3];
#pragma unroll
        for (int g = 0; g < 3; ++g) {
            const int row = g * H + j;
            float a = b_ih[row], b = b_hh[row];
#pragma unroll
            for (int f = 0; f < MAXF; ++f)
                if (f < F) a = fmaf(w_ih[(size_t)row * F + f], x[f], a);
#pragma unroll(SMALL ? HMAX : 4)
            for (int k = 0; k < (SMALL ? HMAX : H); ++k)
                if (!SMALL || k < H) b = fmaf(w_hh[(size_t)row * H + k], h[k], b);
            gi[g] = a;
            gh[g] = b;
        }
        const float r = sigmoidf_ref(__fadd_rn(gh[0], gi[0]));
        const float u = sigmoidf_ref(__fadd_rn(gh[1], gi[1]));
        const float n = tanhf(__fadd_rn(gi[2], __fmul_rn(gh[2], r)));
        hn[j] = __fadd_rn(__fmul_rn(__fsub_rn(h[j], n), u), n);
    }
#pragma unroll
    for (int k = 0; k < MAXA; ++k) z[k] = k < A ? lin_b[k] : 0.0f;
#pragma unroll(SMALL ? HMAX : 1)
    for (int j = 0; j < (SMALL ? HMAX : H); ++j) {
        if (SMALL && j >= H) break;
        h[j] = hn[j];
        const float a = rl_activate(m.act, hn[j]);
#pragma unroll
        for (int k = 0; k < MAXA; ++k)
            if (k < A) z[k] = fmaf(lin_w[(size_t)k * H + j], a, z[k]);
    }
}

// One lstm_cell + activation + Linear for this thread's env (libtorch's lstm_cell, gate order i, f, g, o):
//   gates = (W_ih x + b_ih) + (W_hh h + b_hh);  c' = f c + i g;  h' = o tanh(c')
// c[j] is read and written by unit j alone, so it is updated in place; h waits for all units like grunet_step's.
template <int HMAX, int MAXF, int MAXA>
__device__ __forceinline__ void lstmnet_step(const GruView &m, const float *__restrict__ w, const float *x, float *h, float *c, float *z) {
    const int F = m.F, H = m.H, A = m.A;
    const float *w_ih = w, *w_hh = w_ih + (size_t)4 * H * F, *b_ih = w_hh + (size_t)4 * H * H, *b_hh = b_ih + 4 * H;
    const float *lin_w = b_hh + 4 * H, *lin_b = lin_w + (size_t)A * H;
    constexpr bool SMALL = HMAX <= 8;
    float hn[HMAX];
#pragma unroll(SMALL ? HMAX : 1)
    for (int j = 0; j < (SMALL ? HMAX : H); ++j) {
        if (SMALL && j >= H) break;
        float s[4];
#pragma unroll
        for (int g = 0; g < 4; ++g) {
            const int row = g * H + j;
            float a = b_ih[row], b = b_hh[row];
#pragma unroll
            for (int f = 0; f < MAXF; ++f)
                if (f < F) a = fmaf(w_ih[(size_t)row * F + f], x[f], a);
#pragma unroll(SMALL ? HMAX : 4)
            for (int k = 0; k < (SMALL ? HMAX : H); ++k)
                if (!SMALL || k < H) b = fmaf(w_hh[(size_t)row * H + k], h[k], b);
            s[g] = __fadd_rn(a, b);
        }
        const float i = sigmoidf_ref(s[0]), f = sigmoidf_ref(s[1]), g = tanhf(s[2]), o = sigmoidf_ref(s[3]);
        c[j] = __fadd_rn(__fmul_rn(f, c[j]), __fmul_rn(i, g));
        hn[j] = __fmul_rn(o, tanhf(c[j]));
    }
#pragma unroll
    for (int k = 0; k < MAXA; ++k) z[k] = k < A ? lin_b[k] : 0.0f;
#pragma unroll(SMALL ? HMAX : 1)
    for (int j = 0; j < (SMALL ? HMAX : H); ++j) {
        if (SMALL && j >= H) break;
        h[j] = hn[j];
        const float a = rl_activate(m.act, hn[j]);
#pragma unroll
        for (int k = 0; k < MAXA; ++k)
            if (k < A) z[k] = fmaf(lin_w[(size_t)k * H + j], a, z[k]);
    }
}

// The cell step of a CELL module; c (the LSTM's cell state) is unused by the GRU.
template <int CELL, int HMAX, int MAXF, int MAXA, bool EXACT = false>
__device__ __forceinline__ void seq_step(const GruView &m, const float *__restrict__ w, const float *x, float *h, float *c, float *z) {
    if constexpr (CELL == RL_CELL_LSTM) lstmnet_step<HMAX, MAXF, MAXA>(m, w, x, h, c, z);
    else grunet_step<HMAX, MAXF, MAXA, EXACT>(m, w, x, h, z);
}

struct SeqArgs {
    uint64_t E, lane_offset;
    NoiseSource noise;
    uint32_t min_steps, slack;
    float *obs, *reward, *next_obs;
    uint8_t *action, *succ;
    uint32_t *lane_len;
    uint8_t *lane_flags;
    GruView net;
    int weights_in_smem;
    int F, A;
    double *partials;  // f64 [gridDim.x][ST_COUNT]
    const float *wt;   // K8h only: Wt[F + H][3H]
    int tile_envs;     // K8h only: envs per CTA (32 or 64)
    int stepped;       // K8s: two launches per step, the cell on the tensor cores (gru_step_tc.cuh)
    int eps_greedy;    // the actor: 0 = PolicyActor (categorical on the logits), 1 = DqnActor (epsilon-greedy on the Q-values)
    double eps;        // DqnActor's exploration rate
};

// DqnActor::act (dqn.rs:360-379): gen_bool(eps) on the actor stream, then gen_range(A) when it explores.  The reference returns
// before action_value_fn.step on an explored step, so the caller leaves the episode's hidden state where it was.
template <bool REPLAY>
__device__ __forceinline__ bool dqn_explore(const SeqArgs &a, LaneNoise<REPLAY> &nz, int A, uint32_t &action) {
    if (!rl_gen_bool<REPLAY, RL_STREAM_ACTOR>(nz, a.eps)) return false;
    action = rl_gen_range<REPLAY, RL_STREAM_ACTOR>(nz, (uint32_t)A);
    return true;
}

// XF / XA > 0: features / actions (and hidden = HMAX) fixed at compile time, see grunet_step<EXACT>.  EPS: the epsilon-greedy
// actor of a recurrent Q-network instead of the categorical policy.  CELL: GRU or LSTM (whose cell state c sits beside h).
template <class EnvT, bool REPLAY, int HMAX, bool EPS, int XF = 0, int XA = 0, int CELL = RL_CELL_GRU>
__global__ void __launch_bounds__(128) rollout_seq_kernel(typename EnvT::Params p, SeqArgs a) {
    constexpr bool EXACT = XF > 0;
    constexpr int MF = EXACT ? XF : EnvT::MAXF, MA = EXACT ? XA : EnvT::MAXA;
    auto observe = [&](const typename EnvT::State &st, float *o) {
        if constexpr (EXACT) EnvT::template observe_arms<XA>(st, o);
        else EnvT::observe(p, st, o);
    };
    extern __shared__ __align__(16) float sw[];
    if (a.weights_in_smem) {
        const uint64_t np = a.net.count();
        for (uint64_t i = threadIdx.x; i < np; i += blockDim.x) sw[i] = a.net.params[i];
    }
    __syncthreads();
    const float *w = a.weights_in_smem ? sw : a.net.params;
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid = e < a.E;
    LaneStats st;
    st.init();
    if (valid) {
        const int F = EXACT ? XF : a.F, A = EXACT ? XA : a.A;
        LaneNoise<REPLAY> nz;
        nz.init(a.noise, a.lane_offset + e, e);
        const uint32_t t0 = a.noise.step_counter;
        typename EnvT::State s;
        constexpr int CMAX = CELL == RL_CELL_LSTM ? HMAX : 1;
        float obs[MF], last_obs[MF], h[HMAX], c[CMAX];
#pragma unroll
        for (int f = 0; f < MF; ++f) obs[f] = last_obs[f] = 0.0f;
#pragma unroll
        for (int j = 0; j < HMAX; ++j) h[j] = 0.0f;  // SeqIterative::initial_state (gru.rs:23-28, lstm.rs: (h, c) = 0)
#pragma unroll
        for (int j = 0; j < CMAX; ++j) c[j] = 0.0f;
        uint32_t n = a.min_steps ? a.min_steps + a.slack : 0;  // take_steps.rs:20-31
        uint32_t i = 0;
        int succ_last = RL_TERMINATE, succ_prev = RL_TERMINATE;
        if (n > 0) {  // train.rs:135: every period starts fresh episodes
            nz.set_step(t0);
            EnvT::template reset<REPLAY>(p, s, nz);
            observe(s, obs);
        }
        while (n > 0) {
            nz.set_step(t0 + i);
            float z[MA];
            uint32_t action;
            if (EPS) {
                if (!dqn_explore<REPLAY>(a, nz, A, action)) {
                    seq_step<CELL, HMAX, MF, MA, EXACT>(a.net, w, obs, h, c, z);
                    action = argmax_first<MA>(z, A);
                }
            } else {
                seq_step<CELL, HMAX, MF, MA, EXACT>(a.net, w, obs, h, c, z);
                const float u = rl_u32_to_f32(nz.template next_u32<RL_STREAM_ACTOR>());
                action = categorical_sample<MA>(z, A, u);
            }
#pragma unroll
            for (int f = 0; f < MF; ++f)
                if (f < F) {
                    a.obs[((uint64_t)i * F + f) * a.E + e] = obs[f];
                    last_obs[f] = obs[f];
                }
            float r;
            const int sc = EnvT::template step<REPLAY>(p, s, action, nz, r);
            if (sc == RL_INTERRUPT) {
                observe(s, obs);
#pragma unroll
                for (int f = 0; f < MF; ++f)
                    if (f < F) a.next_obs[((uint64_t)i * F + f) * a.E + e] = obs[f];
            }
            if (sc != RL_CONTINUE) {
                nz.set_step(t0 + i + 1);
                EnvT::template reset<REPLAY>(p, s, nz);
#pragma unroll
                for (int j = 0; j < HMAX; ++j) h[j] = 0.0f;  // steps.rs:116-124: actor.initial_state for the new episode
#pragma unroll
                for (int j = 0; j < CMAX; ++j) c[j] = 0.0f;
            }
            observe(s, obs);
            a.action[(uint64_t)i * a.E + e] = (uint8_t)action;
            a.reward[(uint64_t)i * a.E + e] = r;
            a.succ[(uint64_t)i * a.E + e] = (uint8_t)sc;
            st.push(r, sc);
            succ_prev = succ_last;
            succ_last = sc;
            i += 1;
            n -= 1;
            if (sc != RL_CONTINUE && n <= a.slack) n = 0;  // take_steps.rs:83-88
        }
        const LaneEnd end = finalize_last_episode(i, succ_last, succ_prev);
        if (end.flags & 1u) a.succ[(uint64_t)end.len * a.E + e] = RL_PAD;
        if (end.flags & 2u) {
            a.succ[(uint64_t)(end.len - 1) * a.E + e] = RL_INTERRUPT;
#pragma unroll
            for (int f = 0; f < MF; ++f)
                if (f < F) a.next_obs[((uint64_t)(end.len - 1) * F + f) * a.E + e] = last_obs[f];
        }
        a.lane_len[e] = end.len;
        a.lane_flags[e] = (uint8_t)end.flags;
        st.set_stored(end);
        nz.finish(a.noise, e);
    }
    __shared__ double red[4][ST_COUNT];
    block_reduce_stats(st, valid, red, a.partials);
}

#include "gru_tile.cuh"
#include "gru_step_tc.cuh"

// SeqPacked::seq_packed (gru.rs:72-102 -> chain.rs:157-168) over a stored trajectory: thread per lane, hidden
// state zeroed at the first step of every episode.  out f32 [T][A][E]; PAD slots get zeros.
template <int HMAX, int XF = 0, int XA = 0, int CELL = RL_CELL_GRU>
__global__ void __launch_bounds__(128) grunet_seq_kernel(GruView m, int weights_in_smem, const float *__restrict__ obs,
                                                        const float *__restrict__ next_obs, const uint8_t *__restrict__ succ,
                                                        uint64_t T, uint64_t E, float *__restrict__ out,
                                                        float *__restrict__ out_next) {
    extern __shared__ __align__(16) float sw[];
    if (weights_in_smem) {
        const uint64_t np = m.count();
        for (uint64_t i = threadIdx.x; i < np; i += blockDim.x) sw[i] = m.params[i];
    }
    __syncthreads();
    const float *w = weights_in_smem ? sw : m.params;
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= E) return;
    constexpr bool EXACT = XF > 0;  // sizes fixed at compile time (config 4: 6 features, hidden 4, 1 or 2 outputs)
    constexpr int MAXF = EXACT ? XF : 36, MAXA = EXACT ? XA : 32;
    const int nF = EXACT ? XF : m.F, nA = EXACT ? XA : m.A;
    constexpr int CMAX = CELL == RL_CELL_LSTM ? HMAX : 1;
    float h[HMAX], c[CMAX];
#pragma unroll
    for (int j = 0; j < HMAX; ++j) h[j] = 0.0f;
#pragma unroll
    for (int j = 0; j < CMAX; ++j) c[j] = 0.0f;
    for (uint64_t t = 0; t < T; ++t) {
        const uint8_t sc = succ[t * E + e];
        float z[MAXA];
        if (sc == RL_PAD) {
            for (int k = 0; k < nA; ++k) out[(t * nA + k) * E + e] = 0.0f;
            continue;
        }
        float x[MAXF];
#pragma unroll
        for (int f = 0; f < MAXF; ++f) x[f] = f < nF ? obs[(t * nF + f) * E + e] : 0.0f;
        seq_step<CELL, HMAX, MAXF, MAXA, EXACT>(m, w, x, h, c, z);
        #pragma unroll
        for (int k = 0; k < MAXA; ++k)
            if (k < nA) out[(t * nA + k) * E + e] = z[k];
        if (sc == RL_INTERRUPT && out_next) {
            // the extended observation of an interrupted episode (features.rs:139-185): one more step of the same
            // sequence on the successor observation
            float h2[HMAX], c2[CMAX];
#pragma unroll
            for (int j = 0; j < HMAX; ++j) h2[j] = h[j];
#pragma unroll
            for (int j = 0; j < CMAX; ++j) c2[j] = c[j];
#pragma unroll
            for (int f = 0; f < MAXF; ++f) x[f] = f < nF ? next_obs[(t * nF + f) * E + e] : 0.0f;
            seq_step<CELL, HMAX, MAXF, MAXA, EXACT>(m, w, x, h2, c2, z);
            #pragma unroll
            for (int k = 0; k < MAXA; ++k)
                if (k < nA) out_next[(t * nA + k) * E + e] = z[k];
        }
        if (sc != RL_CONTINUE) {
#pragma unroll
            for (int j = 0; j < HMAX; ++j) h[j] = 0.0f;
#pragma unroll
            for (int j = 0; j < CMAX; ++j) c[j] = 0.0f;
        }
    }
}

GruView view_of(const rl_grunet *g) {
    GruView v;
    v.params = g->params; v.F = g->in_dim; v.H = g->hidden; v.A = g->out_dim; v.act = (int)g->act; v.cell = g->cell;
    return v;
}

constexpr size_t SEQ_SMEM_LIMIT = 160 * 1024;

template <class EnvT, bool REPLAY, int HMAX, bool EPS, int XF, int XA, int CELL>
rl_status launch_seq_k8a(rl_ctx *ctx, const typename EnvT::Params &p, SeqArgs &a, size_t smem, unsigned grid) {
    RL_CUDA(ctx, cudaFuncSetAttribute(rollout_seq_kernel<EnvT, REPLAY, HMAX, EPS, XF, XA, CELL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    RL_LAUNCH(ctx, (rollout_seq_kernel<EnvT, REPLAY, HMAX, EPS, XF, XA, CELL>), grid, 128, smem, p, a);
    return RL_OK;
}

template <class EnvT, int HMAX, int XF = 0, int XA = 0, int CELL = RL_CELL_GRU>
rl_status launch_seq_h(rl_ctx *ctx, const typename EnvT::Params &p, SeqArgs &a, bool replay, size_t smem, unsigned grid) {
    if (a.eps_greedy) {
        if (replay) return launch_seq_k8a<EnvT, true, HMAX, true, XF, XA, CELL>(ctx, p, a, smem, grid);
        return launch_seq_k8a<EnvT, false, HMAX, true, XF, XA, CELL>(ctx, p, a, smem, grid);
    }
    if (replay) return launch_seq_k8a<EnvT, true, HMAX, false, XF, XA, CELL>(ctx, p, a, smem, grid);
    return launch_seq_k8a<EnvT, false, HMAX, false, XF, XA, CELL>(ctx, p, a, smem, grid);
}

template <class EnvT>
rl_status launch_seq(rl_ctx *ctx, const typename EnvT::Params &p, SeqArgs &a, bool replay, size_t smem, unsigned grid) {
    const int H = a.net.H;
    if (a.net.cell == RL_CELL_LSTM) {  // K8a only: the tiled and tensor-core kernels are GRU cells
        if (H <= 8) return launch_seq_h<EnvT, 8, 0, 0, RL_CELL_LSTM>(ctx, p, a, replay, smem, grid);
        return launch_seq_h<EnvT, 128, 0, 0, RL_CELL_LSTM>(ctx, p, a, replay, smem, grid);
    }
    if constexpr (std::is_same<EnvT, BanditMetaEnv>::value) {
        // BASELINE config 4: 2-armed bandit meta-env (6 features) with the rnn.rs-sized GRU (hidden 4)
        if (H == 4 && a.F == 6 && a.A == 2 && p.num_arms == 2) return launch_seq_h<BanditMetaEnv, 4, 6, 2>(ctx, p, a, replay, smem, grid);
    }
    if (H <= 8) return launch_seq_h<EnvT, 8>(ctx, p, a, replay, smem, grid);
    if constexpr (EnvT::MAXA <= GT_LW) {
        if (a.stepped) return launch_seq_stepped<EnvT>(ctx, p, a, replay);       // K8s: hidden 128, cell on tcgen05
        if (a.wt) return launch_seq_tile<EnvT>(ctx, p, a, replay, a.tile_envs);  // K8h: hidden 128
    }
    return launch_seq_h<EnvT, 128>(ctx, p, a, replay, smem, grid);
}

}  // namespace

// Called by rl_rollout (rollout.cu) when the actor carries a sequence network.
rl_status rl_rollout_seq(rl_env *env, rl_grunet *net, bool eps_greedy, double eps, rl_bound bound, rl_traj *traj, double **partials_out,
                         int *nblocks_out) {
    rl_ctx *ctx = env->ctx;
    const rl_env_structure &es = env->structure;
    RL_REQUIRE(ctx, net->ctx == ctx, "rl_rollout: network belongs to another context");
    RL_REQUIRE(ctx, net->in_dim == es.num_features && net->out_dim == es.num_actions,
               "rl_rollout: network dimensions do not match the environment");
    SeqArgs a{};
    a.E = env->E; a.lane_offset = env->lane_offset; a.noise = env->noise;
    a.min_steps = (uint32_t)bound.min_steps; a.slack = (uint32_t)bound.slack_steps;
    a.obs = traj->obs; a.reward = traj->reward; a.next_obs = traj->next_obs; a.action = traj->action; a.succ = traj->succ;
    a.lane_len = traj->lane_len; a.lane_flags = traj->lane_flags;
    a.net = view_of(net);
    a.F = es.num_features; a.A = es.num_actions;
    a.eps_greedy = eps_greedy ? 1 : 0;
    a.eps = eps;
    const size_t wbytes = net->n_params * sizeof(float);
    a.weights_in_smem = wbytes <= SEQ_SMEM_LIMIT;
    const size_t smem = a.weights_in_smem ? wbytes : 16;
    // K8h (gru_tile.cuh) for the rl2-sized module; RL_GRU_KERNEL=thread keeps the thread-per-env kernel (diagnostics)
    const char *pick = getenv("RL_GRU_KERNEL");
    const bool tiled = net->cell == RL_CELL_GRU && net->hidden == GT_H && net->in_dim <= GT_MAXF && net->out_dim <= GT_LW &&
                       env->kind != RL_ENV_MEMORY_GAME && !(pick && strcmp(pick, "thread") == 0);
    a.tile_envs = (pick && strcmp(pick, "tile32") == 0) ? 32 : 64;
    // K8s (gru_step_tc.cuh): the cell of all envs as one tensor-core launch per step.  Picked above 4 096 envs (below, the
    // persistent K8h tile kernel has the shorter step); RL_GRU_KERNEL=stepped / tile / tile32 / thread force a kernel.  K8s
    // serves the categorical policy only: the epsilon-greedy actor takes K8h (tile) wherever K8s would run.
    a.stepped = tiled && !eps_greedy && rl_seq_big_cell_supports(net->in_dim, net->hidden) &&
                ((pick && strcmp(pick, "stepped") == 0) || (!pick && a.E >= 4096));
    const unsigned grid = a.stepped ? rl_grid_for(a.E, 128) : tiled ? (unsigned)((a.E + a.tile_envs - 1) / a.tile_envs) : rl_grid_for(a.E, 128);
    if (tiled && !a.stepped) {
        const size_t wt_floats = (size_t)(net->in_dim + net->hidden) * 3 * net->hidden;
        if (!net->wt) {
            cudaError_t err = cudaMalloc((void **)&net->wt, wt_floats * sizeof(float));
            if (err != cudaSuccess) return rl_fail(ctx, RL_ERR_OOM, "rl_rollout: %s", cudaGetErrorString(err));
        }
        RL_LAUNCH(ctx, gru_wt_kernel, 148, 256, 0, a.net, net->wt);
        a.wt = net->wt;
    }
    double *partials;
    RL_TRY(rl_ctx_scratch(ctx, ((size_t)grid + 1) * ST_COUNT * sizeof(double), (void **)&partials));
    a.partials = partials + ST_COUNT;
    const bool replay = env->noise.mode == RL_NOISE_REPLAY;
    switch (env->kind) {
    case RL_ENV_BANDIT_META: RL_TRY((launch_seq<BanditMetaEnv>(ctx, env->bandit, a, replay, smem, grid))); break;
    case RL_ENV_CARTPOLE: RL_TRY((launch_seq<CartPoleEnv>(ctx, env->cartpole, a, replay, smem, grid))); break;
    case RL_ENV_MEMORY_GAME: RL_TRY((launch_seq<MemoryEnv>(ctx, env->memory, a, replay, smem, grid))); break;
    default: return rl_fail(ctx, RL_ERR_UNSUPPORTED, "rl_rollout: sequence policies are built for the bandit meta-env, MemoryGame and CartPole");
    }
    *partials_out = a.partials;
    *nblocks_out = (int)grid;
    return RL_OK;
}

// SeqPacked forward over a trajectory; out_next (optional) receives the outputs on the successor observation of
// interrupted steps (eval_extended_state_values, critics/mod.rs:116-131).
rl_status rl_grunet_seq_enqueue(rl_grunet *g, rl_traj *traj, float *out_dev, float *out_next_dev) {
    rl_ctx *ctx = g->ctx;
    RL_REQUIRE(ctx, traj->ctx == ctx, "rl_grunet_seq_forward: trajectory belongs to another context");
    RL_REQUIRE(ctx, (int)traj->F == g->in_dim, "rl_grunet_seq_forward: feature count mismatch");
    const uint64_t T = traj->used_T ? traj->used_T : traj->T, E = traj->E;
    const size_t wbytes = g->n_params * sizeof(float);
    const int in_smem = wbytes <= SEQ_SMEM_LIMIT;
    const size_t smem = in_smem ? wbytes : 16;
    const unsigned grid = rl_grid_for(E, 128);
    const GruView v = view_of(g);
    const bool thread = getenv("RL_GRU_KERNEL") && !strcmp(getenv("RL_GRU_KERNEL"), "thread");
    if (g->cell == RL_CELL_LSTM) {
        if (g->hidden > 8 && rl_seq_big_supports(g->in_dim, g->hidden, g->out_dim) && !thread)
            return rl_seq_big_forward(ctx, RL_CELL_LSTM, g->params, g->in_dim, g->hidden, g->out_dim, (int)g->act, traj->obs, traj->next_obs,
                                      traj->succ, T, E, out_dev, out_next_dev);
        if (g->hidden <= 8) {
            RL_CUDA(ctx, cudaFuncSetAttribute(grunet_seq_kernel<8, 0, 0, RL_CELL_LSTM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            RL_LAUNCH(ctx, (grunet_seq_kernel<8, 0, 0, RL_CELL_LSTM>), grid, 128, smem, v, in_smem, traj->obs, traj->next_obs, traj->succ, T, E,
                      out_dev, out_next_dev);
        } else {
            RL_CUDA(ctx, cudaFuncSetAttribute(grunet_seq_kernel<128, 0, 0, RL_CELL_LSTM>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            RL_LAUNCH(ctx, (grunet_seq_kernel<128, 0, 0, RL_CELL_LSTM>), grid, 128, smem, v, in_smem, traj->obs, traj->next_obs, traj->succ, T, E,
                      out_dev, out_next_dev);
        }
        return RL_OK;
    }
    if (g->hidden == 4 && g->in_dim == 6 && (g->out_dim == 1 || g->out_dim == 2)) {
        if (g->out_dim == 1) {
            RL_CUDA(ctx, cudaFuncSetAttribute(grunet_seq_kernel<4, 6, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            RL_LAUNCH(ctx, (grunet_seq_kernel<4, 6, 1>), grid, 128, smem, v, in_smem, traj->obs, traj->next_obs, traj->succ, T, E, out_dev,
                      out_next_dev);
        } else {
            RL_CUDA(ctx, cudaFuncSetAttribute(grunet_seq_kernel<4, 6, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            RL_LAUNCH(ctx, (grunet_seq_kernel<4, 6, 2>), grid, 128, smem, v, in_smem, traj->obs, traj->next_obs, traj->succ, T, E, out_dev,
                      out_next_dev);
        }
    } else if (g->hidden <= 8) {
        RL_CUDA(ctx, cudaFuncSetAttribute(grunet_seq_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        RL_LAUNCH(ctx, grunet_seq_kernel<8>, grid, 128, smem, v, in_smem, traj->obs, traj->next_obs, traj->succ, T, E, out_dev,
                  out_next_dev);
    } else if (rl_seq_big_supports(g->in_dim, g->hidden, g->out_dim) && !thread) {
        // hidden 9 .. 128: the GEMM form (gru_big.cu); the thread-per-lane kernel below stays as the cross-check
        return rl_seq_big_forward(ctx, RL_CELL_GRU, g->params, g->in_dim, g->hidden, g->out_dim, (int)g->act, traj->obs, traj->next_obs, traj->succ, T, E,
                                  out_dev, out_next_dev);
    } else {
        RL_CUDA(ctx, cudaFuncSetAttribute(grunet_seq_kernel<128>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        RL_LAUNCH(ctx, grunet_seq_kernel<128>, grid, 128, smem, v, in_smem, traj->obs, traj->next_obs, traj->succ, T, E, out_dev,
                  out_next_dev);
    }
    return RL_OK;
}

rl_grunet_view rl_grunet_view_of(rl_grunet *g) {
    return rl_grunet_view{g->ctx, g->in_dim, g->hidden, g->out_dim, (int)g->act, g->n_params, g->params, g->cell};
}

namespace {

rl_status seqnet_create(rl_ctx *ctx, int cell, int32_t in_dim, int32_t hidden, int32_t out_dim, rl_activation activation, rl_grunet **out,
                        const char *what) {
    if (!ctx || !out) return rl_fail(ctx, RL_ERR_INVALID_ARG, "%s: NULL argument", what);
    if (!(in_dim >= 1 && in_dim <= 36 && out_dim >= 1 && out_dim <= 32)) return rl_fail(ctx, RL_ERR_INVALID_ARG, "%s: dims out of range", what);
    if (!(hidden >= 1 && hidden <= 128)) return rl_fail(ctx, RL_ERR_INVALID_ARG, "%s: hidden size out of range (1..128)", what);
    RL_CUDA(ctx, cudaSetDevice(ctx->device));
    rl_grunet *g = new (std::nothrow) rl_grunet();
    if (!g) return rl_fail(ctx, RL_ERR_OOM, "%s: host allocation failed", what);
    g->ctx = ctx; g->in_dim = in_dim; g->hidden = hidden; g->out_dim = out_dim; g->act = activation; g->cell = cell;
    g->n_params = view_of(g).count();
    cudaError_t e = cudaMalloc((void **)&g->params, g->n_params * sizeof(float));
    if (e != cudaSuccess) {
        delete g;
        return rl_fail(ctx, RL_ERR_OOM, "%s: %s", what, cudaGetErrorString(e));
    }
    cudaMemsetAsync(g->params, 0, g->n_params * sizeof(float), ctx->stream);
    *out = g;
    return RL_OK;
}

}  // namespace

extern "C" {

rl_status rl_grunet_create(rl_ctx *ctx, int32_t in_dim, int32_t hidden, int32_t out_dim, rl_activation activation,
                           rl_grunet **out) {
    return seqnet_create(ctx, RL_CELL_GRU, in_dim, hidden, out_dim, activation, out, "rl_grunet_create");
}

rl_status rl_lstmnet_create(rl_ctx *ctx, int32_t in_dim, int32_t hidden, int32_t out_dim, rl_activation activation,
                            rl_grunet **out) {
    return seqnet_create(ctx, RL_CELL_LSTM, in_dim, hidden, out_dim, activation, out, "rl_lstmnet_create");
}

rl_status rl_grunet_destroy(rl_grunet *g) {
    if (!g) return RL_OK;
    cudaSetDevice(g->ctx->device);
    cudaStreamSynchronize(g->ctx->stream);
    cudaFree(g->params);
    if (g->wt) cudaFree(g->wt);
    delete g;
    return RL_OK;
}

rl_status rl_grunet_num_params(rl_grunet *g, uint64_t *n) {
    if (!g || !n) return rl_fail(g ? g->ctx : nullptr, RL_ERR_INVALID_ARG, "rl_grunet_num_params: NULL argument");
    *n = g->n_params;
    return RL_OK;
}

rl_status rl_grunet_set_weights(rl_grunet *g, const float *host, uint64_t n) {
    if (!g || !host) return rl_fail(g ? g->ctx : nullptr, RL_ERR_INVALID_ARG, "rl_grunet_set_weights: NULL argument");
    RL_REQUIRE(g->ctx, n == g->n_params, "rl_grunet_set_weights: wrong parameter count");
    RL_CUDA(g->ctx, cudaMemcpyAsync(g->params, host, n * sizeof(float), cudaMemcpyHostToDevice, g->ctx->stream));
    RL_CUDA(g->ctx, cudaStreamSynchronize(g->ctx->stream));
    return RL_OK;
}

rl_status rl_grunet_get_weights(rl_grunet *g, float *host, uint64_t n) {
    if (!g || !host) return rl_fail(g ? g->ctx : nullptr, RL_ERR_INVALID_ARG, "rl_grunet_get_weights: NULL argument");
    RL_REQUIRE(g->ctx, n == g->n_params, "rl_grunet_get_weights: wrong parameter count");
    RL_CUDA(g->ctx, cudaMemcpyAsync(host, g->params, n * sizeof(float), cudaMemcpyDeviceToHost, g->ctx->stream));
    RL_CUDA(g->ctx, cudaStreamSynchronize(g->ctx->stream));
    return RL_OK;
}

rl_status rl_grunet_seq_forward(rl_grunet *g, rl_traj *traj, float *out_dev) {
    if (!g || !traj || !out_dev) return rl_fail(g ? g->ctx : nullptr, RL_ERR_INVALID_ARG, "rl_grunet_seq_forward: NULL argument");
    return rl_grunet_seq_enqueue(g, traj, out_dev, nullptr);
}

}  // extern "C"
