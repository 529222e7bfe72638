// gru_update.cu -- full-batch passes over trajectories for a recurrent policy / critic / Q-network (Chain<Gru, Linear>):
// what autograd does for the reference when the module of Trpo / Ppo / Reinforce / ValuesOpt / DqnAgent is a GRU
// (src/torch/agents/policies/trpo.rs:97-164 with cuDNN disabled :104-108, ppo.rs:97-147, reinforce.rs:64-89, critics/opt.rs:100-127,
// modules/seq/rnn/gru.rs:72-102, modules/chain.rs:157-168).
//
// K9 gru_pass_kernel<MODE>: one thread per lane.  Episodes never cross lanes and a lane's steps are a
// time-ordered column of the [T][.][E] planes, so the recurrence is a plain sequential loop per thread with
// coalesced loads across the warp:
//   forward  t = 0 .. len-1   h_t (stored to hbuf [T][H][E]), logits, per-step loss algebra -> dz_t (dzbuf [T][A][E])
//            MODE = FVP also carries the tangent of h along the direction v (forward-mode R-operator) and
//            stores u_t = (diag p - p p^T) zdot_t instead of a loss gradient
//   backward t = len-1 .. 0   back-propagation through time with dz_t as the output cotangent; the carry is cut
//            at episode boundaries; gates are recomputed from (x_t, h_{t-1})
// The Hessian of mean KL(p0 || p_theta) at theta0 is J^T (diag p - p p^T) J for ANY network (the first-order
// term vanishes at p = p0), so forward-tangent + backward gives exactly the reference's double-backward
// Hessian-vector product.  Per-thread gradients (f32, <= T terms) are summed in f64 in a fixed order into one
// partial row per block, then reduced like the MLP passes (update.cu).
//
// CELL = RL_CELL_LSTM runs the same passes for Chain<Lstm, Linear> (lstm_cell, gate order i, f, g, o): the forward stores
// (h, c) before each step (hbuf, cbuf), FVP carries the tangents (th, tc), BPTT carries (dh, dc), both cut at episode ends:
//   dc = dc_carry + dh' o (1 - tanh^2 c'),  D = (dc g i(1-i), dc c_prev f(1-f), dc i (1-g^2), dh' tanh(c') o(1-o)),
//   dc_carry = dc f,  dh_carry = W_hh^T D.
//
// Sizes: hidden <= 8, features <= 20, actions <= 16 (the rnn.rs-sized and small rl2 bandit modules).  The
// rl2-sized hidden 128 belongs on tensor cores and is not served by this kernel (DESIGN.md section 9).
#include "passes.cuh"

namespace {

constexpr int GH_MAX = 8, GF_MAX = 20, GA_MAX = 16;
constexpr int GP_MAX_ALL = 3 * GH_MAX * GF_MAX + 3 * GH_MAX * GH_MAX + 6 * GH_MAX + GA_MAX * GH_MAX + GA_MAX;

struct Dims {
    int F, H, A, act;
    int NG;  // gates per unit: 3 (GRU) or 4 (LSTM)
    __device__ int o_whh() const { return NG * H * F; }
    __device__ int o_bih() const { return o_whh() + NG * H * H; }
    __device__ int o_bhh() const { return o_bih() + NG * H; }
    __device__ int o_lw() const { return o_bhh() + NG * H; }
    __device__ int o_lb() const { return o_lw() + A * H; }
    __device__ int P() const { return o_lb() + A; }
};

// gates of one gru_cell from (x, h): r, u (update gate, libtorch's "input gate" z), n, and gh_n = W_hn h + b_hn
__device__ __forceinline__ void gru_gates(const Dims &d, const float *__restrict__ w, const float *x, const float *h, float *r,
                                          float *u, float *n, float *ghn) {
    const int F = d.F, H = d.H;
    const float *w_ih = w, *w_hh = w + d.o_whh(), *b_ih = w + d.o_bih(), *b_hh = w + d.o_bhh();
#pragma unroll
    for (int j = 0; j < H; ++j) {
        float gi[3], gh[3];
#pragma unroll
        for (int g = 0; g < 3; ++g) {
            const int row = g * H + j;
            float a = b_ih[row], b = b_hh[row];
#pragma unroll
            for (int f = 0; f < F; ++f) a = fmaf(w_ih[row * F + f], x[f], a);
#pragma unroll
            for (int k = 0; k < H; ++k) b = fmaf(w_hh[row * H + k], h[k], b);
            gi[g] = a;
            gh[g] = b;
        }
        r[j] = sigm(__fadd_rn(gh[0], gi[0]));
        u[j] = sigm(__fadd_rn(gh[1], gi[1]));
        ghn[j] = gh[2];
        n[j] = tanhf(__fadd_rn(gi[2], __fmul_rn(gh[2], r[j])));
    }
}

// activated gates of one lstm_cell from (x, h): i, f, o = sigmoid, g = tanh of (W_ih x + b_ih) + (W_hh h + b_hh)
__device__ __forceinline__ void lstm_gates(const Dims &d, const float *__restrict__ w, const float *x, const float *h, float *ig, float *fg,
                                           float *gg, float *og) {
    const int F = d.F, H = d.H;
    const float *w_ih = w, *w_hh = w + d.o_whh(), *b_ih = w + d.o_bih(), *b_hh = w + d.o_bhh();
#pragma unroll
    for (int j = 0; j < H; ++j) {
        float s[4];
#pragma unroll
        for (int g = 0; g < 4; ++g) {
            const int row = g * H + j;
            float a = b_ih[row], b = b_hh[row];
#pragma unroll
            for (int f = 0; f < F; ++f) a = fmaf(w_ih[row * F + f], x[f], a);
#pragma unroll
            for (int k = 0; k < H; ++k) b = fmaf(w_hh[row * H + k], h[k], b);
            s[g] = __fadd_rn(a, b);
        }
        ig[j] = sigm(s[0]);
        fg[j] = sigm(s[1]);
        gg[j] = tanhf(s[2]);
        og[j] = sigm(s[3]);
    }
}

__device__ __forceinline__ float act_fwd(int act, float v) { return rl_activate(act, v); }

// Back-propagation through time of one lane of an LSTM (len valid steps), accumulating into the per-thread gradient g:
// gates recomputed from (x_t, h_{t-1}, c_{t-1}) stored by the forward, both carries cut at episode ends.
template <int GH, int GF, int GA>
__device__ __forceinline__ void lstm_bptt(const rl_seq_pass_args &a, const Dims &d, const float *__restrict__ sw, float *g, uint64_t len,
                                          uint64_t e) {
    const int F = d.F, H = d.H, A = d.A;
    const uint64_t E = a.E;
    const float *w_hh = sw + d.o_whh(), *lw = sw + d.o_lw();
    float *g_ih = g, *g_hh = g + d.o_whh(), *gb_ih = g + d.o_bih(), *gb_hh = g + d.o_bhh(), *g_lw = g + d.o_lw(), *g_lb = g + d.o_lb();
    float dh[GH], dc[GH];
    for (int j = 0; j < H; ++j) dh[j] = dc[j] = 0.0f;
    for (int64_t t = (int64_t)len - 1; t >= 0; --t) {
        if (a.succ[t * E + e] != RL_CONTINUE)
            for (int j = 0; j < H; ++j) dh[j] = dc[j] = 0.0f;  // last step of its episode: nothing flows back from t + 1
        float x[GF], hp[GH], cp[GH], dz[GA];
        for (int f = 0; f < F; ++f) x[f] = a.obs[(t * F + f) * E + e];
        for (int j = 0; j < H; ++j) {
            hp[j] = a.hbuf[(t * H + j) * E + e];
            cp[j] = a.cbuf[(t * H + j) * E + e];
        }
        for (int k = 0; k < A; ++k) dz[k] = a.dzbuf[(t * A + k) * E + e];
        float ig[GH], fg[GH], gg[GH], og[GH];
        lstm_gates(d, sw, x, hp, ig, fg, gg, og);
        float D[4 * GH], dhp[GH];
        for (int j = 0; j < H; ++j) {
            const float cn = __fadd_rn(__fmul_rn(fg[j], cp[j]), __fmul_rn(ig[j], gg[j]));
            const float tc = tanhf(cn);
            const float hn = __fmul_rn(og[j], tc);
            const float av = act_fwd(d.act, hn);
            float da = 0.0f;
            for (int k = 0; k < A; ++k) {
                da = fmaf(lw[k * H + j], dz[k], da);
                g_lw[k * H + j] = fmaf(dz[k], av, g_lw[k * H + j]);
            }
            const float dhn = fmaf(act_grad(d.act, hn, av), da, dh[j]);
            const float dcn = dc[j] + dhn * og[j] * (1.0f - tc * tc);
            D[j] = dcn * gg[j] * ig[j] * (1.0f - ig[j]);
            D[H + j] = dcn * cp[j] * fg[j] * (1.0f - fg[j]);
            D[2 * H + j] = dcn * ig[j] * (1.0f - gg[j] * gg[j]);
            D[3 * H + j] = dhn * tc * og[j] * (1.0f - og[j]);
            dc[j] = dcn * fg[j];
            dhp[j] = 0.0f;
        }
        for (int k = 0; k < A; ++k) g_lb[k] += dz[k];
        for (int row = 0; row < 4 * H; ++row) {
            const float dg = D[row];
            gb_ih[row] += dg;
            gb_hh[row] += dg;
            for (int f = 0; f < F; ++f) g_ih[row * F + f] = fmaf(dg, x[f], g_ih[row * F + f]);
            for (int k = 0; k < H; ++k) {
                g_hh[row * H + k] = fmaf(dg, hp[k], g_hh[row * H + k]);
                dhp[k] = fmaf(w_hh[row * H + k], dg, dhp[k]);
            }
        }
        for (int j = 0; j < H; ++j) dh[j] = dhp[j];
    }
}

// TF / TH / TA > 0 fix the sizes at compile time (every loop unrolls, every per-thread array -- the 150-odd gradient
// accumulators included -- lives in registers); 0 = sizes from the arguments, arrays of the maximum sizes in local memory.
// CELL: RL_CELL_GRU, or RL_CELL_LSTM (run-time sizes only).  The body stays in the kernel itself: moved into a device
// function behind two kernels, the compile-time-sized GRU instances spilled more (ptxas) and the config-4 update ran 8 % slower.
template <int MODE, int TF, int TH, int TA, int CELL = RL_CELL_GRU>
__global__ void __launch_bounds__(RL_SEQ_BLOCK) gru_pass_kernel(rl_seq_pass_args a) {
    constexpr int GH = TH ? TH : GH_MAX, GF = TF ? TF : GF_MAX, GA = TA ? TA : GA_MAX;
    constexpr bool LSTM = CELL == RL_CELL_LSTM;
    constexpr int NG = rl_cell_gates(CELL), GC = LSTM ? GH : 1;
    constexpr int GP_MAX = NG * GH * GF + NG * GH * GH + 2 * NG * GH + GA * GH + GA;
    using M = PassMode<MODE>;
    constexpr bool BACKWARD = M::BACKWARD, FVP = M::FVP;
    if (a.skip_flag && *a.skip_flag) return;
    const Dims d{TF ? TF : a.F, TH ? TH : a.H, TA ? TA : a.A, a.act, NG};
    const int F = d.F, H = d.H, A = d.A, P = d.P();
    extern __shared__ __align__(16) unsigned char gsm[];
    float *sw = reinterpret_cast<float *>(gsm);      // theta [P]
    float *sv = sw + P;                              // direction [P] (FVP)
#pragma unroll
    for (int i = threadIdx.x; i < P; i += blockDim.x) {
        sw[i] = a.theta[i];
        if (FVP) sv[i] = a.vec[i];
    }
    __syncthreads();
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const bool valid_lane = e < a.E;
    const uint64_t E = a.E;
    float g[BACKWARD ? GP_MAX : 1];
    if (BACKWARD)
        for (int i = 0; i < P; ++i) g[i] = 0.0f;
    double s_loss = 0.0, s_kl = 0.0, s_ent = 0.0, s_cnt = 0.0;

    if (valid_lane) {
        // ---------------- forward ----------------
        float h[GH], hd[GH];
#pragma unroll
        for (int j = 0; j < H; ++j) h[j] = hd[j] = 0.0f;
        float c[GC], cd[GC];
        if constexpr (LSTM)
            for (int j = 0; j < H; ++j) c[j] = cd[j] = 0.0f;
        uint64_t len = 0;
        // software pipeline: the loads of step t + 1 are in flight while step t is computed (a step is ~400 dependent
        // instructions at 2 warps per scheduler: an exposed DRAM latency per step was 35 % of the stall cycles)
        uint8_t sc_next = a.T ? a.succ[e] : (uint8_t)RL_PAD;
        float x_next[GF], tgt_next = 0.0f;
#pragma unroll
        for (int f = 0; f < F; ++f) x_next[f] = a.T ? a.obs[(uint64_t)f * E + e] : 0.0f;
        if (M::USES_TARGET && a.T) tgt_next = a.target[e];
        for (uint64_t t = 0; t < a.T; ++t) {
            const uint8_t sc = sc_next;
            if (sc == RL_PAD) break;
            len = t + 1;
            float x[GF];
#pragma unroll
            for (int f = 0; f < F; ++f) x[f] = x_next[f];
            const float tgt_cur = tgt_next;
            if (t + 1 < a.T) {
                sc_next = a.succ[(t + 1) * E + e];
#pragma unroll
                for (int f = 0; f < F; ++f) x_next[f] = a.obs[((t + 1) * F + f) * E + e];
                if (M::USES_TARGET) tgt_next = a.target[(t + 1) * E + e];
            } else {
                sc_next = RL_PAD;
            }
            if (BACKWARD)
                for (int j = 0; j < H; ++j) a.hbuf[(t * H + j) * E + e] = h[j];
            if constexpr (LSTM)
                if (BACKWARD)
                    for (int j = 0; j < H; ++j) a.cbuf[(t * H + j) * E + e] = c[j];
            float hnew[GH], hdnew[GH], cnew[GC], cdnew[GC];
            if constexpr (LSTM) {
                float ig[GH], fg[GH], gg[GH], og[GH];
                lstm_gates(d, sw, x, h, ig, fg, gg, og);
#pragma unroll
                for (int j = 0; j < H; ++j) {
                    cnew[j] = __fadd_rn(__fmul_rn(fg[j], c[j]), __fmul_rn(ig[j], gg[j]));
                    const float tc = tanhf(cnew[j]);
                    hnew[j] = __fmul_rn(og[j], tc);
                    if (FVP) {
                        // forward-mode tangents along v of the four pre-activations, then of c' and h'
                        const float *v_ih = sv, *v_hh = sv + d.o_whh(), *vb_ih = sv + d.o_bih(), *vb_hh = sv + d.o_bhh();
                        const float *w_hh = sw + d.o_whh();
                        float pd[4];
#pragma unroll
                        for (int q = 0; q < 4; ++q) {
                            const int row = q * H + j;
                            float p = vb_ih[row] + vb_hh[row];
#pragma unroll
                            for (int f = 0; f < F; ++f) p = fmaf(v_ih[row * F + f], x[f], p);
#pragma unroll
                            for (int k = 0; k < H; ++k) p = fmaf(v_hh[row * H + k], h[k], fmaf(w_hh[row * H + k], hd[k], p));
                            pd[q] = p;
                        }
                        const float id = ig[j] * (1.0f - ig[j]) * pd[0], fd = fg[j] * (1.0f - fg[j]) * pd[1];
                        const float gd = (1.0f - gg[j] * gg[j]) * pd[2], od = og[j] * (1.0f - og[j]) * pd[3];
                        cdnew[j] = fd * c[j] + fg[j] * cd[j] + id * gg[j] + ig[j] * gd;
                        hdnew[j] = od * tc + og[j] * (1.0f - tc * tc) * cdnew[j];
                    }
                }
            } else {
            float r[GH], u[GH], n[GH], ghn[GH];
            gru_gates(d, sw, x, h, r, u, n, ghn);
            if (FVP) {
                // forward-mode tangents along v: gi' = V_ih x + v_bih ; gh' = V_hh h + W_hh h' + v_bhh
                const float *v_ih = sv, *v_hh = sv + d.o_whh(), *vb_ih = sv + d.o_bih(), *vb_hh = sv + d.o_bhh();
                const float *w_hh = sw + d.o_whh();
#pragma unroll
                for (int j = 0; j < H; ++j) {
                    float gid[3], ghd[3];
#pragma unroll
                    for (int gg = 0; gg < 3; ++gg) {
                        const int row = gg * H + j;
                        float p = vb_ih[row], q = vb_hh[row];
#pragma unroll
                        for (int f = 0; f < F; ++f) p = fmaf(v_ih[row * F + f], x[f], p);
#pragma unroll
                        for (int k = 0; k < H; ++k) q = fmaf(v_hh[row * H + k], h[k], fmaf(w_hh[row * H + k], hd[k], q));
                        gid[gg] = p;
                        ghd[gg] = q;
                    }
                    const float rd = r[j] * (1.0f - r[j]) * (gid[0] + ghd[0]);
                    const float ud = u[j] * (1.0f - u[j]) * (gid[1] + ghd[1]);
                    const float nd = (1.0f - n[j] * n[j]) * (gid[2] + rd * ghn[j] + r[j] * ghd[2]);
                    hdnew[j] = ud * (h[j] - n[j]) + u[j] * hd[j] + (1.0f - u[j]) * nd;
                }
            }
#pragma unroll
            for (int j = 0; j < H; ++j) hnew[j] = __fadd_rn(__fmul_rn(__fsub_rn(h[j], n[j]), u[j]), n[j]);
            }
            // Chain: activation, Linear
            const float *lw = sw + d.o_lw(), *lb = sw + d.o_lb();
            float z[GA], zd[GA];
#pragma unroll
            for (int k = 0; k < A; ++k) {
                float acc = lb[k], accd = FVP ? sv[d.o_lb() + k] : 0.0f;
#pragma unroll
                for (int j = 0; j < H; ++j) {
                    const float av = act_fwd(d.act, hnew[j]);
                    acc = fmaf(lw[k * H + j], av, acc);
                    if (FVP) accd = fmaf(sv[d.o_lw() + k * H + j], av, fmaf(lw[k * H + j], act_grad(d.act, hnew[j], av) * hdnew[j], accd));
                }
                z[k] = acc;
                zd[k] = accd;
            }
            // ---- per-step loss algebra: the one in passes.cuh, written out over per-thread arrays indexed by run-time values
            // (they live in local memory when the sizes are run-time values).  Routed through sample_loss, whose loops keep
            // such arrays in registers, the run-time-sized GRU Fisher-vector pass went from 64 to 96 registers and the
            // hidden-8 TRPO step ran 30 % slower. ----
            float dz[GA];
#pragma unroll
            for (int k = 0; k < A; ++k) dz[k] = 0.0f;
            float loss_s = 0.0f, kl_s = 0.0f, ent_s = 0.0f;
            const uint64_t n_idx = t * E + e;
            if (M::IS_POLICY) {
                float m = z[0];
#pragma unroll
                for (int k = 1; k < A; ++k) m = fmaxf(m, z[k]);
                float sum = 0.0f;
#pragma unroll
                for (int k = 0; k < A; ++k) sum += expf(z[k] - m);
                const float lse = m + logf(sum);
                float lp[GA], p[GA];
#pragma unroll
                for (int k = 0; k < A; ++k) {
                    lp[k] = z[k] - lse;
                    p[k] = expf(lp[k]);
                }
                const int act_s = (int)a.action[n_idx];
                if (MODE == RL_PASS_STATS) {
#pragma unroll
                    for (int k = 0; k < A; ++k) {
                        ent_s -= fmaxf(lp[k], F32_LOWEST) * p[k];
                        a.logp0[(t * A + k) * E + e] = lp[k];
                    }
                }
                if (M::USES_LP0) {
                    const float lp0a = a.logp0[(t * A + act_s) * E + e];
                    const float ratio = expf(lp[act_s] - lp0a);
                    if (MODE == RL_PASS_PPO) {
                        // -min(ratio adv, clip(ratio) adv); d/d ratio = adv inside [lo, hi] or where the unclipped term is the smaller
                        const float adv_s = a.adv[n_idx];
                        const float clipped = fminf(fmaxf(ratio, a.clip_lo), a.clip_hi);
                        const float t1 = ratio * adv_s, t2 = clipped * adv_s;
                        loss_s = -fminf(t1, t2);
                        const bool inside = ratio >= a.clip_lo && ratio <= a.clip_hi;
                        const float gr = (inside || t1 < t2) ? -t1 : 0.0f;
#pragma unroll
                        for (int k = 0; k < A; ++k) dz[k] = gr * ((act_s == k ? 1.0f : 0.0f) - p[k]);
                    } else {
                        loss_s = -(ratio * a.adv[n_idx]);
#pragma unroll
                        for (int k = 0; k < A; ++k) {
                            const float lp0k = a.logp0[(t * A + k) * E + e];
                            kl_s += fmaxf(lp0k - lp[k], F32_LOWEST) * expf(lp0k);
                            if (MODE == RL_PASS_GRAD) dz[k] = loss_s * ((act_s == k ? 1.0f : 0.0f) - p[k]);
                        }
                    }
                }
                if (MODE == RL_PASS_REINFORCE) {
                    // -(log p(a) adv); the entropy of this evaluation is the one logged (reinforce.rs:72-79)
                    const float adv_s = a.adv[n_idx];
                    loss_s = -(lp[act_s] * adv_s);
#pragma unroll
                    for (int k = 0; k < A; ++k) {
                        ent_s -= fmaxf(lp[k], F32_LOWEST) * p[k];
                        dz[k] = -adv_s * ((act_s == k ? 1.0f : 0.0f) - p[k]);
                    }
                }
                if (FVP) {
                    float pd = 0.0f;
#pragma unroll
                    for (int k = 0; k < A; ++k) pd = fmaf(p[k], zd[k], pd);
#pragma unroll
                    for (int k = 0; k < A; ++k) dz[k] = p[k] * (zd[k] - pd);
                }
            } else if (MODE == RL_PASS_QLOSS) {  // mse(Q(obs).gather(action), targets)  (dqn.rs:316-326)
                const int act_s = (int)a.action[n_idx];
                float q = z[0];
#pragma unroll
                for (int k = 1; k < A; ++k)
                    if (k == act_s) q = z[k];
                const float diff = q - tgt_cur;
                loss_s = diff * diff;
#pragma unroll
                for (int k = 0; k < A; ++k)
                    if (k == act_s) dz[k] = 2.0f * diff;
            } else {  // VALUE: mse(V(obs), targets)  (opt.rs:109-115)
                const float diff = z[0] - tgt_cur;
                loss_s = diff * diff;
                dz[0] = 2.0f * diff;
            }
            s_cnt += 1.0;
            s_loss += (double)loss_s;
            s_kl += (double)kl_s;
            s_ent += (double)ent_s;
            if (BACKWARD)
                for (int k = 0; k < A; ++k) a.dzbuf[(t * A + k) * E + e] = dz[k];
            // next hidden state; a new episode starts from zeros (gru.rs:23-28)
            const bool done = sc != RL_CONTINUE;
#pragma unroll
            for (int j = 0; j < H; ++j) {
                h[j] = done ? 0.0f : hnew[j];
                if (FVP) hd[j] = done ? 0.0f : hdnew[j];
                if constexpr (LSTM) {
                    c[j] = done ? 0.0f : cnew[j];
                    if (FVP) cd[j] = done ? 0.0f : cdnew[j];
                }
            }
        }
        // ---------------- backward (BPTT) ----------------
        if constexpr (LSTM) {
            if (BACKWARD) lstm_bptt<GH, GF, GA>(a, d, sw, g, len, e);
        } else if (BACKWARD) {
            float dh[GH];
#pragma unroll
            for (int j = 0; j < H; ++j) dh[j] = 0.0f;
            const float *w_hh = sw + d.o_whh(), *lw = sw + d.o_lw();
            float *g_ih = g, *g_hh = g + d.o_whh(), *gb_ih = g + d.o_bih(), *gb_hh = g + d.o_bhh(), *g_lw = g + d.o_lw(),
                  *g_lb = g + d.o_lb();
            uint8_t sc_prev = RL_PAD;
            float x_prev[GF], hp_prev[GH], dz_prev[GA];
            auto load_step = [&](uint64_t t) {
                sc_prev = a.succ[t * E + e];
#pragma unroll
                for (int f = 0; f < F; ++f) x_prev[f] = a.obs[(t * F + f) * E + e];
#pragma unroll
                for (int j = 0; j < H; ++j) hp_prev[j] = a.hbuf[(t * H + j) * E + e];
#pragma unroll
                for (int k = 0; k < A; ++k) dz_prev[k] = a.dzbuf[(t * A + k) * E + e];
            };
            if (len > 0) load_step(len - 1);
            for (int64_t t = (int64_t)len - 1; t >= 0; --t) {
                const uint8_t sc = sc_prev;
                if (sc != RL_CONTINUE)
                    for (int j = 0; j < H; ++j) dh[j] = 0.0f;  // last step of its episode: nothing flows back from t + 1
                float x[GF], hp[GH], dz[GA];
#pragma unroll
                for (int f = 0; f < F; ++f) x[f] = x_prev[f];
#pragma unroll
                for (int j = 0; j < H; ++j) hp[j] = hp_prev[j];
#pragma unroll
                for (int k = 0; k < A; ++k) dz[k] = dz_prev[k];
                if (t > 0) load_step((uint64_t)t - 1);  // in flight during this step
                float r[GH], u[GH], n[GH], ghn[GH];
                gru_gates(d, sw, x, hp, r, u, n, ghn);
                float dgi[3 * GH], dgh[3 * GH], dhp[GH];
#pragma unroll
                for (int j = 0; j < H; ++j) {
                    const float hn = __fadd_rn(__fmul_rn(__fsub_rn(hp[j], n[j]), u[j]), n[j]);
                    const float av = act_fwd(d.act, hn);
                    float da = 0.0f;
#pragma unroll
                    for (int k = 0; k < A; ++k) {
                        da = fmaf(lw[k * H + j], dz[k], da);
                        g_lw[k * H + j] = fmaf(dz[k], av, g_lw[k * H + j]);
                    }
                    const float dhn = fmaf(act_grad(d.act, hn, av), da, dh[j]);
                    // h' = u h + (1 - u) n
                    const float du = dhn * (hp[j] - n[j]), dn = dhn * (1.0f - u[j]);
                    dhp[j] = dhn * u[j];
                    const float dpn = dn * (1.0f - n[j] * n[j]);
                    const float dr = dpn * ghn[j];
                    const float dpu = du * u[j] * (1.0f - u[j]);
                    const float dpr = dr * r[j] * (1.0f - r[j]);
                    dgi[j] = dpr; dgi[H + j] = dpu; dgi[2 * H + j] = dpn;
                    dgh[j] = dpr; dgh[H + j] = dpu; dgh[2 * H + j] = dpn * r[j];
                }
#pragma unroll
                for (int k = 0; k < A; ++k) g_lb[k] += dz[k];
#pragma unroll
                for (int row = 0; row < 3 * H; ++row) {
                    const float a_i = dgi[row], a_h = dgh[row];
                    gb_ih[row] += a_i;
                    gb_hh[row] += a_h;
#pragma unroll
                    for (int f = 0; f < F; ++f) g_ih[row * F + f] = fmaf(a_i, x[f], g_ih[row * F + f]);
#pragma unroll
                    for (int k = 0; k < H; ++k) {
                        g_hh[row * H + k] = fmaf(a_h, hp[k], g_hh[row * H + k]);
                        dhp[k] = fmaf(w_hh[row * H + k], a_h, dhp[k]);
                    }
                }
#pragma unroll
                for (int j = 0; j < H; ++j) dh[j] = dhp[j];
            }
        }
    }
    // ---------------- block reduction into one partial row [P + 4] ----------------
    __syncthreads();
    double *part = reinterpret_cast<double *>(gsm);  // reuse: [warps][P + 4]
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, W = P + 4;
    auto wsum = [](double v) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        return v;
    };
    __syncthreads();
    if (BACKWARD) {
#pragma unroll  // static indices keep g[] in registers when the sizes are compile-time
        for (int i = 0; i < P; ++i) {
            const double s = wsum(valid_lane ? (double)g[i] : 0.0);
            if (lane == 0) part[warp * W + i] = s;
        }
    } else {
        for (int i = lane; i < P; i += 32) part[warp * W + i] = 0.0;
    }
    {
        const double v0 = wsum(s_loss), v1 = wsum(s_kl), v2 = wsum(s_ent), v3 = wsum(s_cnt);
        if (lane == 0) {
            part[warp * W + P + 0] = v0; part[warp * W + P + 1] = v1; part[warp * W + P + 2] = v2; part[warp * W + P + 3] = v3;
        }
    }
    __syncthreads();
    double *row = a.partials + (size_t)blockIdx.x * W;
    for (int i = threadIdx.x; i < W; i += blockDim.x) {
        double v = part[i];
#pragma unroll
        for (int w2 = 1; w2 < RL_SEQ_BLOCK / 32; ++w2) v += part[w2 * W + i];
        row[i] = v;
    }
}

template <int MODE, int TF, int TH, int TA, int CELL = RL_CELL_GRU>
rl_status launch_sized(rl_ctx *ctx, const rl_seq_pass_args &a, int grid, size_t smem) {
    RL_CUDA(ctx, cudaFuncSetAttribute(gru_pass_kernel<MODE, TF, TH, TA, CELL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    RL_LAUNCH(ctx, (gru_pass_kernel<MODE, TF, TH, TA, CELL>), grid, RL_SEQ_BLOCK, smem, a);
    return RL_OK;
}

// BASELINE config 4 (2-armed bandit meta-env, rnn.rs-sized GRU): features 6, hidden 4, 2 logits (policy) or 1 (critic)
template <int MODE>
rl_status launch_mode(rl_ctx *ctx, const rl_seq_pass_args &a, int grid, size_t smem) {
    constexpr bool POLICY = MODE != RL_PASS_VALUE;  // the Q-loss pass has one output per action, like a policy
    if (a.cell == RL_CELL_LSTM) return launch_sized<MODE, 0, 0, 0, RL_CELL_LSTM>(ctx, a, grid, smem);
    if (a.F == 6 && a.H == 4 && a.A == (POLICY ? 2 : 1)) return launch_sized<MODE, 6, 4, POLICY ? 2 : 1>(ctx, a, grid, smem);
    return launch_sized<MODE, 0, 0, 0>(ctx, a, grid, smem);
}

}  // namespace

int rl_seq_pass_max_params() { return GP_MAX_ALL; }

bool rl_seq_pass_supports(int F, int H, int A) { return F >= 1 && F <= GF_MAX && H >= 1 && H <= GH_MAX && A >= 1 && A <= GA_MAX; }

// One pass; writes `grid` partial rows of P + 4 doubles (order: loss, kl, entropy, count as in update.cu).
rl_status rl_seq_pass_launch(rl_ctx *ctx, int mode, const rl_seq_pass_args &a, int grid) {
    const int NG = rl_cell_gates(a.cell), P = NG * a.H * a.F + NG * a.H * a.H + 2 * NG * a.H + a.A * a.H + a.A;
    const size_t smem_w = (size_t)2 * P * sizeof(float), smem_r = (size_t)(RL_SEQ_BLOCK / 32) * (P + 4) * sizeof(double);
    const size_t smem = smem_w > smem_r ? smem_w : smem_r;
    switch (mode) {
    case RL_PASS_STATS: return launch_mode<RL_PASS_STATS>(ctx, a, grid, smem);
    case RL_PASS_EVAL: return launch_mode<RL_PASS_EVAL>(ctx, a, grid, smem);
    case RL_PASS_GRAD: return launch_mode<RL_PASS_GRAD>(ctx, a, grid, smem);
    case RL_PASS_FVP: return launch_mode<RL_PASS_FVP>(ctx, a, grid, smem);
    case RL_PASS_VALUE: return launch_mode<RL_PASS_VALUE>(ctx, a, grid, smem);
    case RL_PASS_QLOSS: return launch_mode<RL_PASS_QLOSS>(ctx, a, grid, smem);
    case RL_PASS_PPO: return launch_mode<RL_PASS_PPO>(ctx, a, grid, smem);
    case RL_PASS_REINFORCE: return launch_mode<RL_PASS_REINFORCE>(ctx, a, grid, smem);
    default: return rl_fail(ctx, RL_ERR_INVALID_ARG, "rl_seq_pass_launch: bad mode %d", mode);
    }
}
