// replay.cu -- device-resident ReplayBuffer (one per lane) and the DQN minibatch sampler.
//
// Reference: ReplayBuffer (src/agents/buffers/replay.rs:11-126), finalize_last_episode
// (src/agents/buffers/mod.rs:237-261), DqnAgent::batch_update_slice_refs sample_minibatch
// (src/torch/agents/dqn.rs:280-314), StepValueTarget::targets (src/torch/agents/critics/mod.rs:101-229).
//
// Each lane is one reference worker and owns one ReplayBuffer: a ring of `C` steps from which whole
// oldest episodes are evicted when a step arrives at a full ring.  Layout in HBM (E lanes):
//   obs / next_obs  f32 [E][C][F]   step records of a lane are contiguous, so an episode is one
//   reward          f32 [E][C]      contiguous run (modulo the wrap) and the sampler reads it
//   action, succ    u8  [E][C]      with fully coalesced warp loads
//   ep_end          u32 [E][C]      ring of one-past-the-end SLOTS of the stored episodes
//   total, index_offset u64 [E]; ep_head, ep_count u32 [E]
//
//  K4a replay_book_kernel   thread per lane: the write_step / end_experience bookkeeping (evictions,
//                           episode ends) in step order; copies next_obs of interrupted steps.
//  K4b replay_copy_kernel   [T][P][E] trajectory planes -> [E][C][P] ring through a shared-memory
//                           transpose: coalesced on both sides (HBM bound, 2 x 26 B per step).
//  K4c sample_draw_kernel   thread per draw: round-robin lane, Uniform::new(0, num_episodes) episode.
//  K4d sample_scan_kernel   exclusive scan of the drawn episode lengths, take_while cut (dqn.rs:286-291).
//  K4e sample_gather_kernel warp per sampled episode: ring -> minibatch planes [F][M] + reward-to-go
//                           targets (sequential f32 recurrence, bit-identical to packed.rs:312-342).
//  K4f q_values_kernel / td_target_kernel   OneStepTd: r + gamma * max_a Q(next) (critics/mod.rs:139-151).
//  K4g seq_gather_kernel    the same taken episodes as SEQUENCES for a recurrent Q-network: warp per episode, ring ->
//                           column b of [Lmax][.][B] planes in the trajectory layout (rows past the episode are RL_PAD),
//                           reward-to-go targets by K4e's recurrence.
//  K4h seq_td_target_kernel OneStepTd on the sequence planes from a SeqPacked forward over them.
#include "handles.cuh"

namespace {

enum { RB_ERR_FULL = 1, RB_ERR_NO_EPISODES = 2 };

struct ReplayPtrs {
    uint64_t E, C;
    int F;
    float *obs, *next_obs, *reward;
    uint8_t *action, *succ;
    unsigned long long *total, *index_offset;
    uint32_t *ep_end, *ep_head, *ep_count;
};

__device__ __forceinline__ uint32_t wrap_add(uint32_t a, uint32_t b, uint32_t C) {
    // a < C, b <= C
    const uint64_t s = (uint64_t)a + b;
    return (uint32_t)(s >= C ? s - C : s);
}

// WriteExperienceIncremental::write_step for every step of the lane's thread of experience, then
// end_experience (replay.rs:89-125).  The trajectory already holds the finalised episode (rollout.cu),
// lane_flags says whether a dangling step was dropped (bit 0) and whether the step before it was
// converted to Interrupt (bit 1): the dropped step still went through write_step in the reference and
// may have evicted an episode, and the converted step's episode end is only pushed by end_experience.
__global__ void __launch_bounds__(128)
    replay_book_kernel(ReplayPtrs rb, const uint8_t *__restrict__ succ, const float *__restrict__ next_obs,
                       const uint32_t *__restrict__ lane_len, const uint8_t *__restrict__ lane_flags, uint64_t T,
                       uint32_t *__restrict__ write_start, int *__restrict__ error) {
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= rb.E) return;
    const uint32_t C = (uint32_t)rb.C;
    const uint32_t len = lane_len[e];
    const uint32_t flags = lane_flags[e];
    const bool dropped = flags & 1u, converted = flags & 2u;
    unsigned long long total = rb.total[e], offset = rb.index_offset[e];
    uint32_t head = rb.ep_head[e], count = rb.ep_count[e];
    uint32_t *ends = rb.ep_end + e * rb.C;
    const uint32_t start_slot = (uint32_t)(total % C);
    write_start[e] = start_slot;
    const uint32_t n_raw = len + (dropped ? 1u : 0u);
    uint32_t slot = start_slot;  // slot of the step being written
    bool failed = false;
    for (uint32_t t = 0; t < n_raw; ++t) {
        if (total - offset == C) {  // replay.rs:91-107: full -> drop the oldest episode
            if (count == 0) {       // WriteExperienceError::Full
                failed = true;
                break;
            }
            const uint32_t end_slot = ends[head];
            const uint32_t first = (uint32_t)(offset % C);
            uint32_t ep_len = end_slot >= first ? end_slot - first : end_slot + C - first;
            if (ep_len == 0) ep_len = C;  // an episode that fills the whole ring
            offset += ep_len;
            head = head + 1 == C ? 0 : head + 1;
            count -= 1;
        }
        uint8_t sc = RL_CONTINUE;
        if (t < len) {
            sc = succ[(uint64_t)t * rb.E + e];
            if (converted && t == len - 1) sc = RL_CONTINUE;  // still Continue when it was written
            if (sc == RL_INTERRUPT) {
                for (int f = 0; f < rb.F; ++f)
                    rb.next_obs[(e * rb.C + slot) * rb.F + f] = next_obs[((uint64_t)t * rb.F + f) * rb.E + e];
            }
        }
        total += 1;
        slot = slot + 1 == C ? 0 : slot + 1;
        if (sc != RL_CONTINUE) {  // replay.rs:110-112
            ends[wrap_add(head, count, C)] = slot;
            count += 1;
        }
    }
    if (failed) {
        atomicExch(error, RB_ERR_FULL);
    } else if (dropped) {  // replay.rs:115-125
        total -= 1;
        slot = slot == 0 ? C - 1 : slot - 1;
        if (converted) {
            ends[wrap_add(head, count, C)] = slot;
            count += 1;
            const uint32_t last = slot == 0 ? C - 1 : slot - 1;  // the converted step: Interrupt(dropped observation)
            for (int f = 0; f < rb.F; ++f)
                rb.next_obs[(e * rb.C + last) * rb.F + f] = next_obs[((uint64_t)(len - 1) * rb.F + f) * rb.E + e];
        }
    }
    rb.total[e] = total;
    rb.index_offset[e] = offset;
    rb.ep_head[e] = head;
    rb.ep_count[e] = count;
}

// Transpose NP planes of a [T][NP][E] trajectory array into the [E][C][NP] ring.  A block moves a
// 32-lane x 32-step tile of up to PC planes: loads are coalesced along lanes, stores along (step, plane).
template <typename V, int PC>
__global__ void __launch_bounds__(256)
    replay_copy_kernel(const V *__restrict__ src, V *__restrict__ dst, int NP, uint64_t T, uint64_t E, uint64_t C,
                       const uint32_t *__restrict__ lane_len, const uint32_t *__restrict__ write_start) {
    __shared__ V tile[PC][32][33];
    const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
    const uint64_t e0 = (uint64_t)blockIdx.x * 32;
    const uint32_t t0 = blockIdx.y * 32;
    for (int p0 = 0; p0 < NP; p0 += PC) {
        const int np = NP - p0 < PC ? NP - p0 : PC;
        __syncthreads();
        for (int p = 0; p < np; ++p)
            for (int tt = ty; tt < 32; tt += 8) {
                const uint64_t e = e0 + tx;
                // slots beyond a lane's length are never stored, so no need to mask the load by length
                tile[p][tt][tx] = (e < E && t0 + tt < T) ? src[((uint64_t)(t0 + tt) * NP + p0 + p) * E + e] : V(0);
            }
        __syncthreads();
        for (int le = ty; le < 32; le += 8) {
            const uint64_t e = e0 + le;
            if (e >= E) continue;
            const uint32_t len = lane_len[e], ws = write_start[e];
            for (int idx = tx; idx < 32 * np; idx += 32) {
                const int tt = idx / np, p = idx - tt * np;
                const uint32_t t = t0 + tt;
                if (t < len) {
                    const uint64_t s = ((uint64_t)ws + t) % C;
                    dst[(e * C + s) * NP + p0 + p] = tile[p][tt][le];
                }
            }
        }
    }
}

__global__ void __launch_bounds__(256) replay_stats_kernel(ReplayPtrs rb, unsigned long long *out) {
    unsigned long long s = 0, ep = 0, tot = 0;
    for (uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; e < rb.E; e += (uint64_t)gridDim.x * blockDim.x) {
        s += rb.total[e] - rb.index_offset[e];
        ep += rb.ep_count[e];
        tot += rb.total[e];
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        s += __shfl_xor_sync(0xffffffffu, s, o);
        ep += __shfl_xor_sync(0xffffffffu, ep, o);
        tot += __shfl_xor_sync(0xffffffffu, tot, o);
    }
    if ((threadIdx.x & 31) == 0) {  // integer adds: order does not matter
        atomicAdd(out + 0, s);
        atomicAdd(out + 1, ep);
        atomicAdd(out + 2, tot);
    }
}

// ------------------------------------------------------------------------------------------------
// Minibatch sampling (dqn.rs:280-297)
// ------------------------------------------------------------------------------------------------
struct SampleMeta {
    unsigned long long num_steps;   // M: steps in the minibatch
    unsigned int num_episodes;      // episodes taken
    int error;
    unsigned int max_len;           // longest episode taken (sizes the sequence planes of rl_replay_sample_seq_dev)
};

// Draw j picks buffer j mod E (iter::repeat(buffers).flatten()) and a uniformly random stored episode
// of it: Uniform::new(0, num_episodes).sample (rand 0.8.5 UniformInt::sample, widening multiply with
// rejection zone u64::MAX - (2^64 mod n)).  Philox slot (seed; lane = j, step = draw_index, stream 3).
__global__ void __launch_bounds__(256)
    sample_draw_kernel(ReplayPtrs rb, uint64_t J, uint64_t seed, uint32_t draw_index, uint32_t *__restrict__ sel_lane,
                       uint32_t *__restrict__ sel_start, uint32_t *__restrict__ sel_len, SampleMeta *meta) {
    // blockIdx.y = minibatch of a batched sample (rl_replay_sample_enqueue with n_sets > 1): its own draw index and arrays
    draw_index += blockIdx.y;
    sel_lane += (uint64_t)blockIdx.y * J;
    sel_start += (uint64_t)blockIdx.y * J;
    sel_len += (uint64_t)blockIdx.y * J;
    meta += blockIdx.y;
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= J) return;
    const uint64_t lane = j % rb.E;
    const uint32_t C = (uint32_t)rb.C;
    const uint32_t count = rb.ep_count[lane];
    if (count == 0) {  // Uniform::new(0, 0) panics in the reference
        atomicExch(&meta->error, RB_ERR_NO_EPISODES);
        sel_lane[j] = (uint32_t)lane; sel_start[j] = 0; sel_len[j] = 0;
        return;
    }
    const uint64_t range = count;
    const uint64_t reject = (0xFFFFFFFFFFFFFFFFull - range + 1) % range;
    const uint64_t zone = 0xFFFFFFFFFFFFFFFFull - reject;
    uint32_t k = 0;
    for (uint32_t d = 0; d < 64; ++d) {
        const uint64_t v = rl_philox_slot_impl(seed, j, draw_index, 3, d);
        const uint64_t lo = v * range;
        if (lo <= zone) {
            k = (uint32_t)__umul64hi(v, range);
            break;
        }
    }
    const uint32_t head = rb.ep_head[lane];
    const uint32_t *ends = rb.ep_end + lane * rb.C;
    const uint32_t first = k == 0 ? (uint32_t)(rb.index_offset[lane] % C) : ends[wrap_add(head, k - 1, C)];
    const uint32_t end = ends[wrap_add(head, k, C)];
    uint32_t len = end >= first ? end - first : end + C - first;
    if (len == 0) len = C;
    sel_lane[j] = (uint32_t)lane;
    sel_start[j] = first;
    sel_len[j] = len;
}

// Exclusive scan of the episode lengths in draw order; episodes are taken while the running total is
// below minibatch_steps (take_while, dqn.rs:286-291: the episode that crosses the bound is included).
// One block walks the draws in chunks of 4096 (coalesced uint4 loads, warp + block scan, running carry) and
// stops at the first chunk that starts at or beyond the bound: offsets past the cut are never read.
__global__ void __launch_bounds__(1024)
    sample_scan_kernel(const uint32_t *__restrict__ sel_len, uint64_t J, uint64_t minibatch_steps,
                       unsigned long long *__restrict__ sel_off, SampleMeta *meta) {
    sel_len += (uint64_t)blockIdx.x * J;  // one block per minibatch of a batched sample
    sel_off += (uint64_t)blockIdx.x * J;
    meta += blockIdx.x;
    __shared__ unsigned long long warp_tot[32];
    __shared__ unsigned long long carry_s;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid == 0) carry_s = 0;
    __syncthreads();
    unsigned int taken = 0, longest = 0;
    unsigned long long last_end = 0;
    for (uint64_t base = 0; base < J; base += 4096) {
        const unsigned long long carry = carry_s;
        if (carry >= minibatch_steps) break;  // uniform: every thread reads the same shared value
        const uint64_t j0 = base + (uint64_t)tid * 4;
        uint32_t l[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) l[k] = j0 + k < J ? sel_len[j0 + k] : 0u;
        const unsigned long long mine = (unsigned long long)l[0] + l[1] + l[2] + l[3];
        unsigned long long incl = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const unsigned long long v = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += v;
        }
        if (lane == 31) warp_tot[warp] = incl;
        __syncthreads();
        if (warp == 0) {
            const unsigned long long w = warp_tot[lane];
            unsigned long long wi = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const unsigned long long v = __shfl_up_sync(0xffffffffu, wi, o);
                if (lane >= o) wi += v;
            }
            warp_tot[lane] = wi - w;  // exclusive prefix of the warp totals
            if (lane == 31) carry_s = carry + wi;
        }
        __syncthreads();
        unsigned long long run = carry + warp_tot[warp] + incl - mine;
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            if (j0 + k < J) {
                sel_off[j0 + k] = run;
                if (run < minibatch_steps) {
                    taken += 1;
                    last_end = run + l[k];
                    longest = l[k] > longest ? l[k] : longest;
                }
                run += l[k];
            }
        }
        __syncthreads();  // warp_tot / carry_s are rewritten by the next chunk
    }
    // the taken draws are a prefix, so the counts add up and the largest end is M
    if (taken) {
        atomicAdd(&meta->num_episodes, taken);
        atomicMax(&meta->num_steps, last_end);
        atomicMax(&meta->max_len, longest);
    }
}

struct MinibatchPtrs {
    uint64_t cap;
    float *obs, *nobs, *reward, *target, *qmax, *qmax_next;
    uint8_t *action, *succ, *code;
};

// One warp per sampled episode, walking it from the end in 32-step chunks.
template <bool TD>
__global__ void __launch_bounds__(256)
    sample_gather_kernel(ReplayPtrs rb, const uint32_t *__restrict__ sel_lane, const uint32_t *__restrict__ sel_start,
                         const uint32_t *__restrict__ sel_len, const unsigned long long *__restrict__ sel_off,
                         const SampleMeta *__restrict__ meta, MinibatchPtrs mb, float discount, uint64_t J) {
    {   // blockIdx.y = minibatch of a batched sample: planes of set s start s * cap columns (s * cap * F for obs) further on
        const uint64_t s = blockIdx.y;
        sel_lane += s * J; sel_start += s * J; sel_len += s * J; sel_off += s * J; meta += s;
        mb.obs += s * mb.cap * rb.F; mb.action += s * mb.cap; mb.succ += s * mb.cap; mb.target += s * mb.cap;
        if (TD) { mb.nobs += s * mb.cap * rb.F; mb.reward += s * mb.cap; mb.code += s * mb.cap; }
    }
    const int lane_id = threadIdx.x & 31;
    const uint64_t warp_global = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint64_t total_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const uint32_t n_taken = meta->num_episodes;
    const uint32_t C = (uint32_t)rb.C;
    const int F = rb.F;
    for (uint64_t j = warp_global; j < n_taken; j += total_warps) {
        const uint64_t lane = sel_lane[j];
        const uint32_t start = sel_start[j], len = sel_len[j];
        const uint64_t off = sel_off[j];
        float carry = 0.0f;
        for (int c = (int)((len + 31) / 32) - 1; c >= 0; --c) {
            const uint32_t idx = (uint32_t)c * 32 + lane_id;
            const bool valid = idx < len;
            const uint32_t slot = valid ? wrap_add(start, idx, C) : 0;
            const uint64_t base = lane * rb.C + slot;
            const uint64_t col = off + idx;
            float r = 0.0f;
            uint8_t code = RL_CONTINUE;
            if (valid) {
                r = rb.reward[base];
                code = rb.succ[base];
                if (idx + 1 < len) code = RL_CONTINUE;  // only the last step of the run ends the episode
                mb.action[col] = rb.action[base];
                mb.succ[col] = 0;  // valid sample (anything but RL_PAD)
                for (int f = 0; f < F; ++f) mb.obs[(uint64_t)f * mb.cap + col] = rb.obs[base * F + f];
                if (TD) {
                    mb.reward[col] = r;
                    mb.code[col] = code;
                    if (code == RL_INTERRUPT)
                        for (int f = 0; f < F; ++f) mb.nobs[(uint64_t)f * mb.cap + col] = rb.next_obs[base * F + f];
                }
            }
            if (!TD) {
                // reward_to_go: y_t = x_t + y_{t+1} * d, evaluated strictly in sequence (packed.rs:336)
                const int n_here = (int)(len - (uint32_t)c * 32 < 32u ? len - (uint32_t)c * 32 : 32u);
                float y = 0.0f;
                for (int i = n_here - 1; i >= 0; --i) {
                    const float xi = __shfl_sync(0xffffffffu, r, i);
                    carry = __fadd_rn(xi, __fmul_rn(carry, discount));
                    if (lane_id == i) y = carry;
                }
                if (valid) mb.target[col] = y;
            }
        }
    }
}

// max_a Q(obs) for every minibatch column (and for the successor observation of interrupted steps):
// the BatchMap amax of dqn.rs:300-309 over eval_extended_state_values (critics/mod.rs:116-131).
template <int FT, int AT>
__global__ void __launch_bounds__(256)
    q_values_kernel(MlpView m, MinibatchPtrs mb, const SampleMeta *__restrict__ meta) {
    extern __shared__ float sw[];
    const uint64_t np = m.n_params;
    for (uint64_t i = threadIdx.x; i < np; i += blockDim.x) sw[i] = m.params[i];
    __syncthreads();
    const uint64_t col = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= meta->num_steps) return;
    const int F = m.in_dim, H = m.hidden, A = m.out_dim;
    const float *w1 = sw, *b1 = w1 + (size_t)H * F, *w2 = b1 + H, *b2 = w2 + (size_t)A * H;
    const bool intr = mb.code[col] == RL_INTERRUPT;
    float x[FT], xn[FT], z[AT], zn[AT];
#pragma unroll
    for (int f = 0; f < FT; ++f) {
        x[f] = f < F ? mb.obs[(uint64_t)f * mb.cap + col] : 0.0f;
        xn[f] = (f < F && intr) ? mb.nobs[(uint64_t)f * mb.cap + col] : 0.0f;
    }
#pragma unroll
    for (int k = 0; k < AT; ++k) z[k] = zn[k] = k < A ? b2[k] : 0.0f;
    const bool deep = m.n_hidden > 1;  // MlpConfig::hidden_sizes with two or three entries
    if (deep) {
        rl_mlp_eval_deep(m, sw, x, z);
        if (intr) rl_mlp_eval_deep(m, sw, xn, zn);
    }
    for (int j = 0; j < (deep ? 0 : H); ++j) {
        float acc = b1[j], accn = b1[j];
#pragma unroll
        for (int f = 0; f < FT; ++f)
            if (f < F) {
                const float w = w1[j * F + f];
                acc = fmaf(w, x[f], acc);
                accn = fmaf(w, xn[f], accn);
            }
        const float h = rl_activate(m.act, acc), hn = rl_activate(m.act, accn);
#pragma unroll
        for (int k = 0; k < AT; ++k)
            if (k < A) {
                z[k] = fmaf(w2[k * H + j], h, z[k]);
                zn[k] = fmaf(w2[k * H + j], hn, zn[k]);
            }
    }
    float best = z[0], bestn = zn[0];
#pragma unroll
    for (int k = 1; k < AT; ++k)
        if (k < A) {
            best = fmaxf(best, z[k]);
            bestn = fmaxf(bestn, zn[k]);
        }
    mb.qmax[col] = best;
    if (intr) mb.qmax_next[col] = bestn;
}

// one_step_values: rewards + discount * estimated_next_values (critics/mod.rs:139-151); the value after
// a terminal step is 0 (masked_fill_ of the invalid extended observation, critics/mod.rs:127-129).
__global__ void __launch_bounds__(256)
    td_target_kernel(MinibatchPtrs mb, const SampleMeta *__restrict__ meta, float discount) {
    const uint64_t col = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (col >= meta->num_steps) return;
    const uint8_t code = mb.code[col];
    const float next = code == RL_CONTINUE ? mb.qmax[col + 1] : code == RL_INTERRUPT ? mb.qmax_next[col] : 0.0f;
    mb.target[col] = __fadd_rn(mb.reward[col], __fmul_rn(discount, next));
}

// Sequence planes of one sample: B = episodes taken (one column each, in draw order), L = the longest of them.
struct SeqPlanes {
    uint64_t B, L;
    float *obs, *nobs, *reward, *target, *qout, *qout_next;  // obs / nobs f32 [L][F][B]; reward, target [L][B]; q* [L][A][B]
    uint8_t *action, *succ;                                  // u8 [L][B]
    uint32_t *len;                                           // u32 [B] episode lengths
};

// One warp per taken episode, walking it from the end in 32-step chunks like sample_gather_kernel: step idx of draw j goes to
// row idx of column j.  The reward-to-go carry is the same sequential f32 recurrence, so the targets are bit-identical to the
// flat minibatch's.  Column j's successor codes are RL_CONTINUE up to the last step, which keeps the stored code.
__global__ void __launch_bounds__(256)
    seq_gather_kernel(ReplayPtrs rb, const uint32_t *__restrict__ sel_lane, const uint32_t *__restrict__ sel_start,
                      const uint32_t *__restrict__ sel_len, SeqPlanes sp, float discount, int rtg) {
    const int lane_id = threadIdx.x & 31;
    const uint64_t warp_global = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint64_t total_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const uint32_t C = (uint32_t)rb.C;
    const int F = rb.F;
    const uint64_t B = sp.B;
    for (uint64_t j = warp_global; j < B; j += total_warps) {
        const uint64_t lane = sel_lane[j];
        const uint32_t start = sel_start[j], len = sel_len[j];
        if (lane_id == 0) sp.len[j] = len;
        float carry = 0.0f;
        for (int c = (int)((len + 31) / 32) - 1; c >= 0; --c) {
            const uint32_t idx = (uint32_t)c * 32 + lane_id;
            const bool valid = idx < len;
            const uint64_t base = lane * rb.C + (valid ? wrap_add(start, idx, C) : 0);
            const uint64_t cell = (uint64_t)idx * B + j;
            float r = 0.0f;
            if (valid) {
                r = rb.reward[base];
                const uint8_t code = idx + 1 < len ? (uint8_t)RL_CONTINUE : rb.succ[base];
                sp.reward[cell] = r;
                sp.action[cell] = rb.action[base];
                sp.succ[cell] = code;
                for (int f = 0; f < F; ++f) sp.obs[((uint64_t)idx * F + f) * B + j] = rb.obs[base * F + f];
                if (code == RL_INTERRUPT)
                    for (int f = 0; f < F; ++f) sp.nobs[((uint64_t)idx * F + f) * B + j] = rb.next_obs[base * F + f];
            }
            if (rtg) {  // packed.rs:336, as in sample_gather_kernel
                const int n_here = (int)(len - (uint32_t)c * 32 < 32u ? len - (uint32_t)c * 32 : 32u);
                float y = 0.0f;
                for (int i = n_here - 1; i >= 0; --i) {
                    const float xi = __shfl_sync(0xffffffffu, r, i);
                    carry = __fadd_rn(xi, __fmul_rn(carry, discount));
                    if (lane_id == i) y = carry;
                }
                if (valid) sp.target[cell] = y;
            }
        }
    }
}

// one_step_values on the sequence planes (critics/mod.rs:139-151) from Q = seq_packed over them (qout) and Q on the successor
// observation of the interrupted last steps (qout_next, one more step of the same sequence): the operations of q_values_kernel's
// max and td_target_kernel's sum, in the same order.
__global__ void __launch_bounds__(256) seq_td_target_kernel(SeqPlanes sp, int A, float discount) {
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x, B = sp.B;
    if (i >= sp.L * B) return;
    const uint64_t t = i / B, b = i - t * B;
    const uint8_t code = sp.succ[i];
    if (code == RL_PAD) return;
    auto qmax = [&](const float *q, uint64_t row) {
        float best = q[(row * A) * B + b];
        for (int k = 1; k < A; ++k) best = fmaxf(best, q[(row * A + k) * B + b]);
        return best;
    };
    const float next = code == RL_CONTINUE ? qmax(sp.qout, t + 1) : code == RL_INTERRUPT ? qmax(sp.qout_next, t) : 0.0f;
    sp.target[i] = __fadd_rn(sp.reward[i], __fmul_rn(discount, next));
}

}  // namespace

struct rl_replay {
    rl_ctx *ctx = nullptr;
    rl_env *env = nullptr;
    ReplayPtrs p{};
    uint32_t *write_start = nullptr;
    int *error = nullptr;
    unsigned long long *stats = nullptr;
    // sampler state
    uint64_t mb_minibatch = 0;
    uint32_t mb_sets = 0;  // minibatches the sampler arrays hold (batched sampling of a whole update)
    MinibatchPtrs mb{};
    uint32_t *sel_lane = nullptr, *sel_start = nullptr, *sel_len = nullptr;
    unsigned long long *sel_off = nullptr;
    SampleMeta *meta = nullptr;        // single-sample meta (rl_replay_create)
    SampleMeta *meta_sets = nullptr;   // [mb_sets] for batched samples
    uint32_t last_sets = 1;            // minibatches of the last enqueue (rl_replay_sample_finish reads the last one)
    uint32_t draw_counter = 0;
    // sequence sampler (rl_replay_sample_seq_dev): planes grown to the largest B * L seen, and the rl_traj that views them
    SeqPlanes seq{};
    uint64_t seq_cells = 0, seq_cols = 0;
    int seq_A = 0;
    rl_traj seq_traj{};
};

namespace {

void free_seq(rl_replay *rb) {
    SeqPlanes &q = rb->seq;
    cudaFree(q.obs); cudaFree(q.nobs); cudaFree(q.reward); cudaFree(q.target); cudaFree(q.qout); cudaFree(q.qout_next);
    cudaFree(q.action); cudaFree(q.succ); cudaFree(q.len);
    q = SeqPlanes{};
    rb->seq_cells = rb->seq_cols = 0;
    rb->seq_A = 0;
}

// Planes for `cells` = B * L steps and B columns (A outputs of the Q-network for OneStepTd targets, 0 = none), grown only.
rl_status ensure_seq(rl_replay *rb, uint64_t cells, uint64_t cols, int A) {
    rl_ctx *ctx = rb->ctx;
    if (cells <= rb->seq_cells && cols <= rb->seq_cols && A <= rb->seq_A) return RL_OK;
    RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    cells = cells > rb->seq_cells ? cells : rb->seq_cells;
    cols = cols > rb->seq_cols ? cols : rb->seq_cols;
    A = A > rb->seq_A ? A : rb->seq_A;
    free_seq(rb);
    const size_t F = (size_t)rb->p.F;
    SeqPlanes &q = rb->seq;
    cudaError_t e = cudaSuccess;
    auto alloc = [&](void **p, size_t bytes) {
        if (e == cudaSuccess && bytes) e = cudaMalloc(p, bytes);
    };
    alloc((void **)&q.obs, cells * F * sizeof(float));
    alloc((void **)&q.nobs, cells * F * sizeof(float));
    alloc((void **)&q.reward, cells * sizeof(float));
    alloc((void **)&q.target, cells * sizeof(float));
    alloc((void **)&q.qout, cells * (size_t)A * sizeof(float));
    alloc((void **)&q.qout_next, cells * (size_t)A * sizeof(float));
    alloc((void **)&q.action, cells);
    alloc((void **)&q.succ, cells);
    alloc((void **)&q.len, cols * sizeof(uint32_t));
    if (e != cudaSuccess) {
        free_seq(rb);
        return rl_fail(ctx, RL_ERR_OOM, "replay sequence sampler: %s", cudaGetErrorString(e));
    }
    rb->seq_cells = cells;
    rb->seq_cols = cols;
    rb->seq_A = A;
    return RL_OK;
}

void free_sampler(rl_replay *rb) {
    cudaFree(rb->mb.obs); cudaFree(rb->mb.nobs); cudaFree(rb->mb.reward); cudaFree(rb->mb.target);
    cudaFree(rb->mb.qmax); cudaFree(rb->mb.qmax_next); cudaFree(rb->mb.action); cudaFree(rb->mb.succ);
    cudaFree(rb->mb.code); cudaFree(rb->sel_lane); cudaFree(rb->sel_start); cudaFree(rb->sel_len);
    cudaFree(rb->sel_off);
    rb->mb = MinibatchPtrs{};
    rb->sel_lane = rb->sel_start = rb->sel_len = nullptr;
    rb->sel_off = nullptr;
    rb->mb_minibatch = 0;
    rb->mb_sets = 0;
    cudaFree(rb->meta_sets);
    rb->meta_sets = nullptr;
}

rl_status ensure_sampler(rl_replay *rb, uint64_t minibatch_steps, uint32_t sets, bool td) {
    rl_ctx *ctx = rb->ctx;
    if (rb->mb_minibatch == minibatch_steps && rb->mb.obs && rb->mb_sets >= sets && (!td || rb->mb.nobs)) return RL_OK;
    RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    free_sampler(rb);
    // the last episode taken may overshoot the bound by at most one ring of steps
    const uint64_t cap = ((minibatch_steps + rb->p.C + 1 + 31) / 32) * 32;
    const size_t F = (size_t)rb->p.F, S = sets;
    cudaError_t e = cudaSuccess;
    auto alloc = [&](void **p, size_t bytes) {
        if (e == cudaSuccess) e = cudaMalloc(p, bytes);
    };
    alloc((void **)&rb->mb.obs, S * cap * F * sizeof(float));
    alloc((void **)&rb->mb.target, S * cap * sizeof(float));
    alloc((void **)&rb->mb.action, S * cap);
    alloc((void **)&rb->mb.succ, S * cap);
    if (td) {  // OneStepTd targets only (sampled one minibatch at a time: they depend on the current parameters)
        alloc((void **)&rb->mb.nobs, cap * F * sizeof(float));
        alloc((void **)&rb->mb.reward, cap * sizeof(float));
        alloc((void **)&rb->mb.qmax, cap * sizeof(float));
        alloc((void **)&rb->mb.qmax_next, cap * sizeof(float));
        alloc((void **)&rb->mb.code, cap);
    }
    alloc((void **)&rb->sel_lane, S * minibatch_steps * sizeof(uint32_t));
    alloc((void **)&rb->sel_start, S * minibatch_steps * sizeof(uint32_t));
    alloc((void **)&rb->sel_len, S * minibatch_steps * sizeof(uint32_t));
    alloc((void **)&rb->sel_off, S * minibatch_steps * sizeof(unsigned long long));
    alloc((void **)&rb->meta_sets, S * sizeof(SampleMeta));
    if (e != cudaSuccess) {
        free_sampler(rb);
        return rl_fail(ctx, RL_ERR_OOM, "replay sampler: %s", cudaGetErrorString(e));
    }
    rb->mb.cap = cap;
    rb->mb_minibatch = minibatch_steps;
    rb->mb_sets = sets;
    return RL_OK;
}

}  // namespace

// Enqueue `n_sets` sample_minibatch calls (dqn.rs:280-314) with draw indices draw_index .. draw_index + n_sets - 1 on
// the context stream; no host synchronisation.  The ring does not change during an update and reward-to-go targets
// do not depend on the parameters, so the minibatches of all optimizer steps of one update are drawn, cut and
// gathered by three launches (grid.y = minibatch) -- large enough to run at HBM speed -- and come out exactly as
// n_sets separate calls would produce them.  Set s starts s * capacity columns after set 0 in every plane.
// OneStepTd targets need the parameters of their step: n_sets must be 1.
rl_status rl_replay_sample_enqueue(rl_replay *rb, uint64_t minibatch_steps, uint64_t seed, uint32_t draw_index,
                                   int one_step_td, float discount, rl_mlp *q, uint32_t n_sets, rl_minibatch_dev *out) {
    rl_ctx *ctx = rb->ctx;
    RL_REQUIRE(ctx, minibatch_steps > 0 && minibatch_steps < (1ull << 31), "replay sample: minibatch_steps out of range");
    RL_REQUIRE(ctx, n_sets >= 1 && n_sets <= 65535 && (!one_step_td || n_sets == 1), "replay sample: bad number of minibatches");
    RL_TRY(ensure_sampler(rb, minibatch_steps, n_sets, one_step_td != 0));
    SampleMeta *meta = rb->meta_sets;
    if (one_step_td) {
        RL_REQUIRE(ctx, q != nullptr, "replay sample: OneStepTd targets need the action-value network");
        RL_REQUIRE(ctx, q->in_dim == rb->p.F, "replay sample: network input does not match the observation features");
        RL_REQUIRE(ctx, q->in_dim <= 36 && q->out_dim <= 32, "replay sample: network too large");
    }
    const uint64_t J = minibatch_steps;  // every episode has at least one step
    RL_CUDA(ctx, cudaMemsetAsync(meta, 0, (size_t)n_sets * sizeof(SampleMeta), ctx->stream));
    RL_CUDA(ctx, cudaMemsetAsync(rb->mb.succ, RL_PAD, (size_t)n_sets * rb->mb.cap, ctx->stream));
    RL_LAUNCH(ctx, sample_draw_kernel, dim3(rl_grid_for(J, 256), n_sets), 256, 0, rb->p, J, seed, draw_index, rb->sel_lane,
              rb->sel_start, rb->sel_len, meta);
    RL_LAUNCH(ctx, sample_scan_kernel, n_sets, 1024, 0, rb->sel_len, J, minibatch_steps, rb->sel_off, meta);
    const dim3 gather_grid(n_sets > 1 ? (unsigned)ctx->sm_count : (unsigned)ctx->sm_count * 4, n_sets);
    if (one_step_td) {
        RL_LAUNCH(ctx, sample_gather_kernel<true>, gather_grid, 256, 0, rb->p, rb->sel_lane, rb->sel_start, rb->sel_len,
                  rb->sel_off, meta, rb->mb, discount, J);
        const size_t smem = q->n_params * sizeof(float);
        const unsigned grid = rl_grid_for(rb->mb.cap, 256);
        if (q->in_dim <= 8 && q->out_dim <= 2) {
            RL_CUDA(ctx, cudaFuncSetAttribute(q_values_kernel<8, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            RL_LAUNCH(ctx, (q_values_kernel<8, 2>), grid, 256, smem, rl_mlp_view(q), rb->mb, meta);
        } else {
            if (q->in_dim > 36 || q->out_dim > 32)
                return rl_fail(ctx, RL_ERR_UNSUPPORTED, "replay sample: one-step TD targets are built for <= 36 features and <= 32 actions");
            RL_CUDA(ctx, cudaFuncSetAttribute(q_values_kernel<36, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            RL_LAUNCH(ctx, (q_values_kernel<36, 32>), grid, 256, smem, rl_mlp_view(q), rb->mb, meta);
        }
        RL_LAUNCH(ctx, td_target_kernel, grid, 256, 0, rb->mb, meta, discount);
    } else {
        RL_LAUNCH(ctx, sample_gather_kernel<false>, gather_grid, 256, 0, rb->p, rb->sel_lane, rb->sel_start, rb->sel_len,
                  rb->sel_off, meta, rb->mb, discount, J);
    }
    rb->last_sets = n_sets;
    out->capacity = rb->mb.cap;
    out->obs = rb->mb.obs;
    out->action = rb->mb.action;
    out->target = rb->mb.target;
    out->succ = rb->mb.succ;
    return RL_OK;
}

// Check the device-side error flag of the last sample (synchronises).
rl_status rl_replay_sample_finish(rl_replay *rb, uint64_t *num_steps, uint64_t *num_episodes) {
    rl_ctx *ctx = rb->ctx;
    SampleMeta *host;
    const uint32_t sets = rb->last_sets ? rb->last_sets : 1;
    RL_REQUIRE(ctx, rb->meta_sets != nullptr, "replay sample: nothing was sampled");
    RL_TRY(rl_ctx_pinned(ctx, (size_t)sets * sizeof(SampleMeta), (void **)&host));
    RL_CUDA(ctx, cudaMemcpyAsync(host, rb->meta_sets, (size_t)sets * sizeof(SampleMeta), cudaMemcpyDeviceToHost, ctx->stream));
    RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    for (uint32_t i = 0; i < sets; ++i)
        if (host[i].error == RB_ERR_NO_EPISODES)
            return rl_fail(ctx, RL_ERR_INVALID_ARG, "replay sample: a lane has no stored episode (Uniform::new(0, 0))");
    if (num_steps) *num_steps = host[sets - 1].num_steps;
    if (num_episodes) *num_episodes = host[sets - 1].num_episodes;
    return RL_OK;
}

// sample_minibatch (dqn.rs:280-314) for a recurrent Q-network: K4c / K4d exactly as rl_replay_sample_enqueue draws and cuts
// them (same episodes), then the taken episodes as padded sequences in an rl_traj of B lanes and L steps that the recurrent
// passes and forwards read like a rollout's trajectory.  B and L are known only on the device: one host read of the sample's
// SampleMeta sizes the planes, so this call synchronises.  OneStepTd targets need `q` (a SeqPacked forward with the current
// parameters); reward-to-go targets do not.
rl_status rl_replay_sample_seq_dev(rl_replay *rb, uint64_t minibatch_steps, uint64_t seed, uint32_t draw_index, int one_step_td,
                                   float discount, rl_grunet *q, rl_traj **out_traj, const float **out_target) {
    rl_ctx *ctx = rb->ctx;
    RL_REQUIRE(ctx, minibatch_steps > 0 && minibatch_steps < (1ull << 31), "replay sample: minibatch_steps out of range");
    rl_grunet_view qv{};
    if (one_step_td) {
        RL_REQUIRE(ctx, q != nullptr, "replay sample: OneStepTd targets need the action-value network");
        qv = rl_grunet_view_of(q);
        RL_REQUIRE(ctx, qv.ctx == ctx, "replay sample: network belongs to another context");
        RL_REQUIRE(ctx, qv.in_dim == rb->p.F, "replay sample: network input does not match the observation features");
    }
    RL_TRY(ensure_sampler(rb, minibatch_steps, 1, false));
    SampleMeta *meta = rb->meta_sets;
    const uint64_t J = minibatch_steps;
    RL_CUDA(ctx, cudaMemsetAsync(meta, 0, sizeof(SampleMeta), ctx->stream));
    RL_LAUNCH(ctx, sample_draw_kernel, dim3(rl_grid_for(J, 256), 1), 256, 0, rb->p, J, seed, draw_index, rb->sel_lane, rb->sel_start,
              rb->sel_len, meta);
    RL_LAUNCH(ctx, sample_scan_kernel, 1, 1024, 0, rb->sel_len, J, minibatch_steps, rb->sel_off, meta);
    rb->last_sets = 1;
    SampleMeta *host;
    RL_TRY(rl_ctx_pinned(ctx, sizeof(SampleMeta), (void **)&host));
    RL_CUDA(ctx, cudaMemcpyAsync(host, meta, sizeof(SampleMeta), cudaMemcpyDeviceToHost, ctx->stream));
    RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (host->error == RB_ERR_NO_EPISODES)
        return rl_fail(ctx, RL_ERR_INVALID_ARG, "replay sample: a lane has no stored episode (Uniform::new(0, 0))");
    const uint64_t B = host->num_episodes, L = host->max_len, M = host->num_steps;
    RL_TRY(ensure_seq(rb, B * L, B, one_step_td ? qv.out_dim : 0));
    SeqPlanes sp = rb->seq;
    sp.B = B;
    sp.L = L;
    rb->seq.B = B;
    rb->seq.L = L;
    RL_CUDA(ctx, cudaMemsetAsync(sp.succ, RL_PAD, B * L, ctx->stream));
    // padded rows are read by the GEMM form of the passes (multiplied by zero cotangents): keep them finite
    RL_CUDA(ctx, cudaMemsetAsync(sp.obs, 0, B * L * (size_t)rb->p.F * sizeof(float), ctx->stream));
    RL_LAUNCH(ctx, seq_gather_kernel, (unsigned)ctx->sm_count * 4, 256, 0, rb->p, rb->sel_lane, rb->sel_start, rb->sel_len, sp, discount,
              one_step_td ? 0 : 1);
    rl_traj &t = rb->seq_traj;
    t.ctx = ctx; t.env = rb->env;
    t.E = B; t.T = L; t.used_T = L; t.F = (uint64_t)rb->p.F;
    t.obs = sp.obs; t.reward = sp.reward; t.next_obs = sp.nobs; t.action = sp.action; t.succ = sp.succ;
    t.lane_len = sp.len; t.lane_flags = nullptr; t.counts_dev = nullptr;
    t.num_steps = M; t.num_episodes = B;
    if (one_step_td) {
        RL_TRY(rl_grunet_seq_enqueue(q, &t, sp.qout, sp.qout_next));
        RL_LAUNCH(ctx, seq_td_target_kernel, rl_grid_for(B * L, 256), 256, 0, sp, qv.out_dim, discount);
    }
    *out_traj = &t;
    *out_target = sp.target;
    return RL_OK;
}

uint32_t rl_replay_next_draw_index(rl_replay *rb) { return rb->draw_counter++; }
uint32_t rl_replay_take_draw_indices(rl_replay *rb, uint32_t n) {
    const uint32_t first = rb->draw_counter;
    rb->draw_counter += n;
    return first;
}
rl_ctx *rl_replay_ctx(rl_replay *rb) { return rb->ctx; }
int rl_replay_num_features(rl_replay *rb) { return rb->p.F; }

extern "C" {

rl_status rl_replay_create(rl_env *env, uint64_t step_capacity_per_lane, rl_replay **out) {
    if (!env || !out) return rl_fail(env ? env->ctx : nullptr, RL_ERR_INVALID_ARG, "rl_replay_create: NULL argument");
    rl_ctx *ctx = env->ctx;
    *out = nullptr;
    RL_REQUIRE(ctx, step_capacity_per_lane >= 1 && step_capacity_per_lane < (1ull << 31),
               "rl_replay_create: capacity out of range");
    RL_CUDA(ctx, cudaSetDevice(ctx->device));
    rl_replay *rb = new (std::nothrow) rl_replay();
    if (!rb) return rl_fail(ctx, RL_ERR_OOM, "rl_replay_create: host allocation failed");
    rb->ctx = ctx;
    rb->env = env;
    ReplayPtrs &p = rb->p;
    p.E = env->E; p.C = step_capacity_per_lane; p.F = env->structure.num_features;
    const size_t EC = (size_t)p.E * p.C;
    cudaError_t e = cudaSuccess;
    auto alloc = [&](void **ptr, size_t bytes) {
        if (e == cudaSuccess) e = cudaMalloc(ptr, bytes);
    };
    alloc((void **)&p.obs, EC * p.F * sizeof(float));
    alloc((void **)&p.next_obs, EC * p.F * sizeof(float));
    alloc((void **)&p.reward, EC * sizeof(float));
    alloc((void **)&p.action, EC);
    alloc((void **)&p.succ, EC);
    alloc((void **)&p.ep_end, EC * sizeof(uint32_t));
    alloc((void **)&p.total, p.E * sizeof(unsigned long long));
    alloc((void **)&p.index_offset, p.E * sizeof(unsigned long long));
    alloc((void **)&p.ep_head, p.E * sizeof(uint32_t));
    alloc((void **)&p.ep_count, p.E * sizeof(uint32_t));
    alloc((void **)&rb->write_start, p.E * sizeof(uint32_t));
    alloc((void **)&rb->error, sizeof(int));
    alloc((void **)&rb->stats, 4 * sizeof(unsigned long long));
    alloc((void **)&rb->meta, sizeof(SampleMeta));
    if (e != cudaSuccess) {
        rl_replay_destroy(rb);
        return rl_fail(ctx, e == cudaErrorMemoryAllocation ? RL_ERR_OOM : RL_ERR_CUDA, "rl_replay_create: %s",
                       cudaGetErrorString(e));
    }
    cudaMemsetAsync(p.total, 0, p.E * sizeof(unsigned long long), ctx->stream);
    cudaMemsetAsync(p.index_offset, 0, p.E * sizeof(unsigned long long), ctx->stream);
    cudaMemsetAsync(p.ep_head, 0, p.E * sizeof(uint32_t), ctx->stream);
    cudaMemsetAsync(p.ep_count, 0, p.E * sizeof(uint32_t), ctx->stream);
    cudaMemsetAsync(rb->error, 0, sizeof(int), ctx->stream);
    *out = rb;
    return RL_OK;
}

rl_status rl_replay_destroy(rl_replay *rb) {
    if (!rb) return RL_OK;
    cudaSetDevice(rb->ctx->device);
    cudaStreamSynchronize(rb->ctx->stream);
    ReplayPtrs &p = rb->p;
    cudaFree(p.obs); cudaFree(p.next_obs); cudaFree(p.reward); cudaFree(p.action); cudaFree(p.succ);
    cudaFree(p.ep_end); cudaFree(p.total); cudaFree(p.index_offset); cudaFree(p.ep_head); cudaFree(p.ep_count);
    cudaFree(rb->write_start); cudaFree(rb->error); cudaFree(rb->stats); cudaFree(rb->meta);
    free_sampler(rb);
    free_seq(rb);
    delete rb;
    return RL_OK;
}

rl_status rl_replay_append(rl_replay *rb, rl_traj *traj) {
    if (!rb || !traj) return rl_fail(rb ? rb->ctx : nullptr, RL_ERR_INVALID_ARG, "rl_replay_append: NULL argument");
    rl_ctx *ctx = rb->ctx;
    RL_REQUIRE(ctx, traj->env == rb->env, "rl_replay_append: trajectory belongs to another env");
    const uint64_t T = traj->used_T ? traj->used_T : traj->T, E = rb->p.E;
    if (T == 0) return RL_OK;
    RL_LAUNCH(ctx, replay_book_kernel, rl_grid_for(E, 128), 128, 0, rb->p, traj->succ, traj->next_obs, traj->lane_len,
              traj->lane_flags, T, rb->write_start, rb->error);
    const dim3 grid(rl_div_up(E, 32), rl_div_up(T, 32));
    RL_LAUNCH(ctx, (replay_copy_kernel<float, 8>), grid, 256, 0, traj->obs, rb->p.obs, rb->p.F, T, E, rb->p.C,
              traj->lane_len, rb->write_start);
    RL_LAUNCH(ctx, (replay_copy_kernel<float, 1>), grid, 256, 0, traj->reward, rb->p.reward, 1, T, E, rb->p.C,
              traj->lane_len, rb->write_start);
    RL_LAUNCH(ctx, (replay_copy_kernel<uint8_t, 1>), grid, 256, 0, traj->action, rb->p.action, 1, T, E, rb->p.C,
              traj->lane_len, rb->write_start);
    RL_LAUNCH(ctx, (replay_copy_kernel<uint8_t, 1>), grid, 256, 0, traj->succ, rb->p.succ, 1, T, E, rb->p.C,
              traj->lane_len, rb->write_start);
    int *host;
    RL_TRY(rl_ctx_pinned(ctx, sizeof(int), (void **)&host));
    RL_CUDA(ctx, cudaMemcpyAsync(host, rb->error, sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (*host == RB_ERR_FULL) {
        cudaMemsetAsync(rb->error, 0, sizeof(int), ctx->stream);
        return rl_fail(ctx, RL_ERR_BUFFER_FULL,
                       "rl_replay_append: an episode does not fit the per-lane capacity of %llu steps (WriteExperienceError::Full)",
                       (unsigned long long)rb->p.C);
    }
    return RL_OK;
}

rl_status rl_replay_stats_of(rl_replay *rb, rl_replay_stats *out) {
    if (!rb || !out) return rl_fail(rb ? rb->ctx : nullptr, RL_ERR_INVALID_ARG, "rl_replay_stats_of: NULL argument");
    rl_ctx *ctx = rb->ctx;
    RL_CUDA(ctx, cudaMemsetAsync(rb->stats, 0, 4 * sizeof(unsigned long long), ctx->stream));
    const unsigned grid = rl_div_up(rb->p.E, 256) < 1024u ? rl_div_up(rb->p.E, 256) : 1024u;
    RL_LAUNCH(ctx, replay_stats_kernel, grid, 256, 0, rb->p, rb->stats);
    unsigned long long *host;
    RL_TRY(rl_ctx_pinned(ctx, 4 * sizeof(unsigned long long), (void **)&host));
    RL_CUDA(ctx, cudaMemcpyAsync(host, rb->stats, 3 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    out->num_steps = host[0];
    out->num_episodes = host[1];
    out->total_step_count = host[2];
    return RL_OK;
}

rl_status rl_replay_read_lane(rl_replay *rb, uint64_t lane, uint64_t max_steps, float *obs_host, uint8_t *action_host,
                              float *reward_host, uint8_t *succ_host, float *next_obs_host, uint64_t *episode_len_host,
                              rl_replay_stats *lane_stats) {
    if (!rb || !lane_stats) return rl_fail(rb ? rb->ctx : nullptr, RL_ERR_INVALID_ARG, "rl_replay_read_lane: NULL argument");
    rl_ctx *ctx = rb->ctx;
    const ReplayPtrs &p = rb->p;
    RL_REQUIRE(ctx, lane < p.E, "rl_replay_read_lane: lane out of range");
    unsigned long long total, offset;
    uint32_t head, count;
    RL_CUDA(ctx, cudaMemcpyAsync(&total, p.total + lane, 8, cudaMemcpyDeviceToHost, ctx->stream));
    RL_CUDA(ctx, cudaMemcpyAsync(&offset, p.index_offset + lane, 8, cudaMemcpyDeviceToHost, ctx->stream));
    RL_CUDA(ctx, cudaMemcpyAsync(&head, p.ep_head + lane, 4, cudaMemcpyDeviceToHost, ctx->stream));
    RL_CUDA(ctx, cudaMemcpyAsync(&count, p.ep_count + lane, 4, cudaMemcpyDeviceToHost, ctx->stream));
    RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    const uint64_t n = total - offset;
    lane_stats->num_steps = n;
    lane_stats->num_episodes = count;
    lane_stats->total_step_count = total;
    RL_REQUIRE(ctx, n <= max_steps, "rl_replay_read_lane: host arrays too small");
    const uint64_t first = offset % p.C;
    // the stored steps are [first, first + n) modulo C: at most two contiguous runs
    const uint64_t run0 = n < p.C - first ? n : p.C - first, run1 = n - run0;
    auto copy = [&](void *dst, const void *src_base, size_t elem) -> cudaError_t {
        if (!dst) return cudaSuccess;
        const char *src = (const char *)src_base + (size_t)lane * p.C * elem;
        cudaError_t e = cudaMemcpyAsync(dst, src + first * elem, run0 * elem, cudaMemcpyDeviceToHost, ctx->stream);
        if (e == cudaSuccess && run1)
            e = cudaMemcpyAsync((char *)dst + run0 * elem, src, run1 * elem, cudaMemcpyDeviceToHost, ctx->stream);
        return e;
    };
    RL_CUDA(ctx, copy(obs_host, p.obs, (size_t)p.F * sizeof(float)));
    RL_CUDA(ctx, copy(next_obs_host, p.next_obs, (size_t)p.F * sizeof(float)));
    RL_CUDA(ctx, copy(reward_host, p.reward, sizeof(float)));
    RL_CUDA(ctx, copy(action_host, p.action, 1));
    RL_CUDA(ctx, copy(succ_host, p.succ, 1));
    RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
    if (episode_len_host && count) {
        std::string tmp;
        tmp.resize((size_t)p.C * sizeof(uint32_t));
        uint32_t *ends = (uint32_t *)&tmp[0];
        RL_CUDA(ctx, cudaMemcpyAsync(ends, p.ep_end + lane * p.C, (size_t)p.C * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
        RL_CUDA(ctx, cudaStreamSynchronize(ctx->stream));
        uint64_t prev = first;
        for (uint32_t k = 0; k < count; ++k) {
            const uint64_t end = ends[(head + k) % p.C];
            uint64_t len = end >= prev ? end - prev : end + p.C - prev;
            if (len == 0) len = p.C;
            episode_len_host[k] = len;
            prev = end;
        }
    }
    return RL_OK;
}

double rl_exploration_rate(double start, double end, uint64_t period, uint64_t global_steps, int32_t training) {
    // ExplorationRateSchedule::exploration_rate (schedules.rs:35-45)
    if (!training) return 0.0;
    if (period == 0) return end;
    double frac = (double)global_steps / (double)period;
    if (frac > 1.0) frac = 1.0;
    return frac * (end - start) + start;
}

rl_status rl_replay_sample(rl_replay *rb, const rl_dqn_cfg *cfg, rl_mlp *q, uint32_t draw_index, rl_minibatch_view *out) {
    if (!rb || !cfg || !out) return rl_fail(rb ? rb->ctx : nullptr, RL_ERR_INVALID_ARG, "rl_replay_sample: NULL argument");
    rl_minibatch_dev dev{};
    RL_TRY(rl_replay_sample_enqueue(rb, cfg->minibatch_steps, cfg->sample_seed, draw_index, cfg->target_one_step_td,
                                    cfg->discount_factor, q, 1, &dev));
    uint64_t m = 0, eps = 0;
    RL_TRY(rl_replay_sample_finish(rb, &m, &eps));
    out->num_steps = m;
    out->num_episodes = eps;
    out->capacity = dev.capacity;
    out->obs = dev.obs;
    out->action = dev.action;
    out->target = dev.target;
    out->succ = dev.succ;
    return RL_OK;
}

rl_status rl_replay_sample_seq(rl_replay *rb, const rl_dqn_cfg *cfg, rl_grunet *q, uint32_t draw_index, rl_traj_view *out,
                               const float **target_dev) {
    if (!rb || !cfg || !out || !target_dev)
        return rl_fail(rb ? rb->ctx : nullptr, RL_ERR_INVALID_ARG, "rl_replay_sample_seq: NULL argument");
    rl_traj *t = nullptr;
    RL_TRY(rl_replay_sample_seq_dev(rb, cfg->minibatch_steps, cfg->sample_seed, draw_index, cfg->target_one_step_td,
                                    cfg->discount_factor, q, &t, target_dev));
    RL_CUDA(rb->ctx, cudaStreamSynchronize(rb->ctx->stream));
    out->num_lanes = t->E; out->step_capacity = t->T; out->num_features = t->F;
    out->obs = t->obs; out->action = t->action; out->reward = t->reward; out->succ = t->succ; out->next_obs = t->next_obs;
    out->lane_len = t->lane_len;
    out->num_steps = t->num_steps;
    return RL_OK;
}

}  // extern "C"
