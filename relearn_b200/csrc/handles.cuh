// handles.cuh -- definitions of the opaque C-ABI handles, shared between translation units.
#pragma once

#include "common.cuh"
#include "envs.cuh"

struct rl_env {
    rl_ctx *ctx = nullptr;
    rl_env_kind kind = RL_ENV_CARTPOLE;
    uint64_t E = 0, lane_offset = 0;
    CartPoleEnv::Params cartpole{};
    ChainEnv::Params chain{};
    MemoryEnv::Params memory{};
    BanditMetaEnv::Params bandit{};
    PartitionEnv::Params partition{};
    rl_env_structure structure{};
    EnvStatePtrs state{};
    NoiseSource noise{};
    // outputs of the unfused step
    float *obs = nullptr, *reward = nullptr, *next_obs = nullptr;
    uint8_t *succ = nullptr;
};

// MlpConfig::hidden_sizes (mlp.rs:25-34): one hidden layer takes the specialised kernels; two or three take the
// layer-generic paths (rl_mlp_eval_deep below, mlp_pass_any_kernel's DEEP form in update.cu).
constexpr int RL_MLP_MAX_HIDDEN_LAYERS = 3, RL_DEEP_MAXH = 256;

struct rl_mlp {
    rl_ctx *ctx = nullptr;
    int in_dim = 0, hidden = 0, out_dim = 0;  // hidden = hid[0]
    int n_hidden = 1, hid[RL_MLP_MAX_HIDDEN_LAYERS] = {0, 0, 0};
    rl_activation act = RL_ACT_RELU;
    uint64_t n_params = 0;
    float *params = nullptr;  // device, flat in Module::variables() order
    __host__ __device__ static uint64_t count(int in, int hidden, int out) {
        return (uint64_t)hidden * in + hidden + (uint64_t)out * hidden + out;
    }
    // [W, b] per Linear, layers in order (mlp.rs:126-128)
    __host__ __device__ static uint64_t count_layers(int in, const int *hid, int n_hidden, int out) {
        uint64_t n = 0;
        int prev = in;
        for (int l = 0; l < n_hidden; ++l) {
            n += (uint64_t)hid[l] * prev + hid[l];
            prev = hid[l];
        }
        return n + (uint64_t)out * prev + out;
    }
};

struct rl_adam {
    const void *owner = nullptr;  // the module handle this optimizer was built for (rl_mlp* or rl_grunet*)
    rl_ctx *ctx = nullptr;
    rl_adam_cfg cfg{};
    float *m = nullptr, *v = nullptr;  // device, n_params each
    uint64_t step = 0;
};

struct rl_traj {
    rl_ctx *ctx = nullptr;
    rl_env *env = nullptr;
    uint64_t E = 0, T = 0, F = 0;
    float *obs = nullptr, *reward = nullptr, *next_obs = nullptr;
    uint8_t *action = nullptr, *succ = nullptr;
    uint32_t *lane_len = nullptr;
    uint8_t *lane_flags = nullptr;  // bit 0: dangling step dropped, bit 1: previous step converted to Interrupt
    uint64_t num_steps = 0;     // valid steps (host copy, refreshed by rollout / load)
    uint64_t num_episodes = 0;
    uint64_t used_T = 0;        // number of time slots in use (<= T)
    double *counts_dev = nullptr;  // device: [0] = num_steps, [1] = num_episodes (f64 for all-reduce)
};

// Minibatch planes produced by the replay sampler (replay.cu), consumed by rl_dqn_update (update.cu).
struct rl_minibatch_dev {
    uint64_t capacity;       // columns allocated (valid ones have succ != RL_PAD)
    const float *obs;        // f32 [F][capacity]
    const uint8_t *action;   // u8 [capacity]
    const float *target;     // f32 [capacity]
    const uint8_t *succ;     // u8 [capacity]
};
// n_sets minibatches with consecutive draw indices; set s starts s * capacity columns (s * capacity * F for obs) after
// set 0 in every plane
rl_status rl_replay_sample_enqueue(rl_replay *rb, uint64_t minibatch_steps, uint64_t seed, uint32_t draw_index,
                                   int one_step_td, float discount, rl_mlp *q, uint32_t n_sets, rl_minibatch_dev *out);
uint32_t rl_replay_take_draw_indices(rl_replay *rb, uint32_t n);
rl_status rl_replay_sample_finish(rl_replay *rb, uint64_t *num_steps, uint64_t *num_episodes);
uint32_t rl_replay_next_draw_index(rl_replay *rb);
rl_ctx *rl_replay_ctx(rl_replay *rb);
int rl_replay_num_features(rl_replay *rb);
// The same draws as sequences for a recurrent Q-network (replay.cu K4g / K4h): *out_traj views B = episodes taken lanes of
// L = the longest episode's steps (valid until the next sequence sample on this buffer), *out_target f32 [L][B].  Synchronises.
rl_status rl_replay_sample_seq_dev(rl_replay *rb, uint64_t minibatch_steps, uint64_t seed, uint32_t draw_index, int one_step_td,
                                   float discount, rl_grunet *q, rl_traj **out_traj, const float **out_target);

// The cell of a recurrent module (rl_grunet_create / rl_lstmnet_create); the kernel selectors below read it.
enum { RL_CELL_GRU = 0, RL_CELL_LSTM = 1 };
__host__ __device__ constexpr int rl_cell_gates(int cell) { return cell == RL_CELL_LSTM ? 4 : 3; }
struct rl_grunet_view { rl_ctx *ctx; int in_dim, hidden, out_dim, act; uint64_t n_params; float *params; int cell; };
rl_grunet_view rl_grunet_view_of(rl_grunet *g);
rl_status rl_grunet_seq_enqueue(rl_grunet *g, rl_traj *traj, float *out_dev, float *out_next_dev);

// Full-batch pass modes shared by the MLP passes (update.cu) and the recurrent passes (gru_update.cu)
enum { RL_PASS_STATS = 0, RL_PASS_EVAL = 1, RL_PASS_GRAD = 2, RL_PASS_FVP = 3, RL_PASS_VALUE = 4, RL_PASS_QLOSS = 5,
       RL_PASS_PPO = 6, RL_PASS_REINFORCE = 7 };

// Arguments of one recurrent pass (gru_update.cu).  Scratch planes are [T][.][E] like the trajectory.
struct rl_seq_pass_args {
    const float *obs;
    const uint8_t *action, *succ;
    uint64_t T, E;
    int F, H, A, act;
    const float *theta, *vec, *adv, *target;
    float *logp0;   // f32 [T][A][E]
    float *hbuf;    // f32 [T][H][E]  hidden state before each step
    float *dzbuf;   // f32 [T][A][E]  output cotangent of each step
    double *partials;
    const int *skip_flag;
    int cell;       // RL_CELL_GRU / RL_CELL_LSTM
    float *cbuf;    // f32 [T][H][E]  LSTM: cell state before each step (K9)
    float clip_lo, clip_hi;  // RL_PASS_PPO: 1 -+ clip_distance as f32 (ppo.rs:131-132)
};
// lanes per block (= per partial row) of the recurrent passes: two warps, so that a block's warps finish close together
constexpr int RL_SEQ_BLOCK = 64;
rl_status rl_seq_pass_launch(rl_ctx *ctx, int mode, const rl_seq_pass_args &a, int grid);
bool rl_seq_pass_supports(int F, int H, int A);
// gru_big.cu (K10): the same passes as tiled GEMMs over the lanes of a step, hidden <= 128; ONE partial row at a.partials
bool rl_seq_big_supports(int F, int H, int A);
rl_status rl_seq_big_pass_launch(rl_ctx *ctx, int mode, const rl_seq_pass_args &a);
// one gru_cell over all lanes on the tensor cores (hidden 128) for the stepped rollout K8s (gru.cu)
bool rl_seq_big_cell_supports(int F, int H);
size_t rl_seq_big_prepared_bytes(int F, int H);
rl_status rl_seq_big_prepare(rl_ctx *ctx, const float *params, int F, int H, void *prepared);
rl_status rl_seq_big_cell(rl_ctx *ctx, const void *prepared, int F, int H, const float *x, const float *h, uint64_t E, float *hnew);
rl_status rl_seq_big_forward(rl_ctx *ctx, int cell, const float *params, int F, int H, int A, int act, const float *obs,
                             const float *next_obs, const uint8_t *succ, uint64_t T, uint64_t E, float *out, float *out_next);

// gru.cu: fused rollout with a recurrent policy.  *partials_out receives the device pointer of its *nblocks_out rows of
// per-block statistics (steps.cuh: ST_COUNT sums each), with one more row in front of them for the totals; rl_rollout
// sums them as it does for every rollout.
// eps_greedy selects DqnActor (epsilon-greedy on the Q-values, exploration rate eps) instead of PolicyActor.
rl_status rl_rollout_seq(rl_env *env, rl_grunet *net, bool eps_greedy, double eps, rl_bound bound, rl_traj *traj, double **partials_out,
                         int *nblocks_out);

struct rl_tabq {
    rl_ctx *ctx = nullptr;
    uint64_t R = 0;
    int S = 0, A = 0;
    double discount = 1.0;
    double *q = nullptr;        // f64 [R][S][A]
    unsigned long long *counts = nullptr;  // u64 [R][S][A]
};

struct rl_ucb1 {
    rl_ctx *ctx = nullptr;
    uint64_t R = 0;
    int S = 0, A = 0;
    double rate = 0.2, scale = 1.0, shift = 0.0;  // exploration_rate; reward_scale_factor, reward_shift (ucb.rs:118-123)
    double *mean = nullptr;                  // f64 [R][S][A]
    unsigned long long *count = nullptr;     // u64 [R][S][A]
    unsigned long long *visits = nullptr;    // u64 [R][S]
};

struct rl_bts {
    rl_ctx *ctx = nullptr;
    uint64_t R = 0;
    int S = 0, A = 0;
    int num_samples = 1;
    double threshold = 0.0;                  // (reward_min + reward_max) / 2 (thompson_sampling.rs:102-103)
    unsigned long long *low = nullptr;       // u64 [R][S][A]
    unsigned long long *high = nullptr;      // u64 [R][S][A]
};

// Mlp weights passed by value into kernels
struct MlpView {
    const float *params;
    int in_dim, hidden, out_dim, act;
    int n_hidden, hid[RL_MLP_MAX_HIDDEN_LAYERS];
    uint32_t n_params;
    __device__ const float *w1() const { return params; }
    __device__ const float *b1() const { return params + (size_t)hidden * in_dim; }
    __device__ const float *w2() const { return b1() + hidden; }
    __device__ const float *b2() const { return w2() + (size_t)out_dim * hidden; }
};

// Shared-memory layout of an Mlp for the warp-cooperative kernels (update.cu's run-time-sized passes, rollout.cu's
// warp-per-env rollout): every Linear's weights TRANSPOSED as [input][unit] with an odd row pitch, so that a sweep with the
// lanes over units (fixed input) and a sweep with the lanes over inputs (fixed unit) are both conflict-free.
struct DeepLayout {
    int n_layers;                  // Linear layers = hidden layers + 1
    int in[4], out[4], ld[4];      // per Linear: inputs, units, pitch (odd)
    int off_w[4], off_b[4];        // offsets in the padded layout
    int nat_w[4];                  // offsets in Module::variables() order
    int P, P_pad, maxH;
};
__host__ __device__ inline DeepLayout rl_mlp_layout(int F, int L, const int *Hs, int A) {
    DeepLayout d{};
    d.n_layers = L + 1;
    int prev = F, off = 0, nat = 0, maxH = 0;
    for (int l = 0; l <= L; ++l) {
        const int out = l < L ? Hs[l] : A;
        d.in[l] = prev; d.out[l] = out; d.ld[l] = out | 1;
        d.off_w[l] = off; off += prev * d.ld[l];
        d.off_b[l] = off; off += out;
        d.nat_w[l] = nat; nat += prev * out + out;
        if (l < L && out > maxH) maxH = out;
        prev = out;
    }
    d.P = nat; d.P_pad = off; d.maxH = maxH;
    return d;
}
// natural parameter index -> index in the padded transposed layout
__host__ __device__ inline int deep_pidx(const DeepLayout &d, int i) {
    for (int l = 0; l < d.n_layers; ++l) {
        const int r = i - d.nat_w[l], nw = d.in[l] * d.out[l];
        if (r < nw) return d.off_w[l] + (r % d.in[l]) * d.ld[l] + r / d.in[l];
        if (r < nw + d.out[l]) return d.off_b[l] + (r - nw);
    }
    return 0;
}

inline MlpView rl_mlp_view(const rl_mlp *m) {
    MlpView v;
    v.params = m ? m->params : nullptr;
    v.in_dim = m ? m->in_dim : 0;
    v.hidden = m ? m->hidden : 0;
    v.out_dim = m ? m->out_dim : 0;
    v.act = m ? (int)m->act : 0;
    v.n_hidden = m ? m->n_hidden : 1;
    for (int l = 0; l < RL_MLP_MAX_HIDDEN_LAYERS; ++l) v.hid[l] = m ? m->hid[l] : 0;
    v.n_params = m ? (uint32_t)m->n_params : 0u;
    return v;
}

__device__ __forceinline__ float rl_activate(int act, float v) {
    switch (act) {
    case RL_ACT_RELU: return v < 0.0f ? 0.0f : v;  // NaN propagates like torch.relu
    case RL_ACT_SIGMOID: return 1.0f / (1.0f + expf(-v));
    case RL_ACT_TANH: return tanhf(v);
    default: return v;
    }
}

// Mlp::forward (mlp.rs:139-151) for one input on one thread, two or three hidden layers: x[in_dim] -> z[out_dim].
// `w` is the flat parameter vector (shared or global memory).  Activations ping-pong through two local arrays; the
// one-hidden-layer modules never come here (their kernels stream the hidden units without storing them).
static __device__ __noinline__ void rl_mlp_eval_deep(const MlpView &m, const float *w, const float *x, float *z) {
    float ha[RL_DEEP_MAXH], hb[RL_DEEP_MAXH];
    const float *in = x;
    int n_in = m.in_dim;
    for (int l = 0; l < m.n_hidden; ++l) {
        float *out = (l & 1) ? hb : ha;
        const int H = m.hid[l];
        const float *W = w, *b = w + (size_t)H * n_in;
        for (int j = 0; j < H; ++j) {
            float acc = b[j];
            for (int f = 0; f < n_in; ++f) acc = fmaf(W[(size_t)j * n_in + f], in[f], acc);
            out[j] = rl_activate(m.act, acc);
        }
        w = b + H;
        in = out;
        n_in = H;
    }
    const float *W = w, *b = w + (size_t)m.out_dim * n_in;
    for (int k = 0; k < m.out_dim; ++k) {
        float acc = b[k];
        for (int f = 0; f < n_in; ++f) acc = fmaf(W[(size_t)k * n_in + f], in[f], acc);
        z[k] = acc;
    }
}
