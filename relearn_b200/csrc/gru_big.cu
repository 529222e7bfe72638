// gru_big.cu -- K10: the full-batch passes of the update for a recurrent module of ANY hidden size up to 128
// (Chain<Gru(F -> H), act, Linear(H -> A)>, the rl2-sized policy / critic of relearn_experiments/src/bin/rl2-bandits.rs:379-451),
// as tiled GEMMs over all lanes of a time step.  Same contract as gru_pass_kernel (gru_update.cu, hidden <= 8, one thread
// per lane): a partial row [P + 4] of f64 sums -- gradient or Fisher-vector product, loss, KL, entropy, count -- that
// update.cu reduces over the data-parallel group and feeds to the trust-region step / Adam.
//
// What autograd does for the reference (trpo.rs:97-164 with cuDNN disabled :104-108, critics/opt.rs:100-127,
// modules/seq/rnn/gru.rs:72-102), restated as batched linear algebra on the [T][.][E] planes of the trajectory:
//
//   forward, t = 0 .. T-1   G_t [4H x E] = Wc [4H x (F + H)] . [x_t ; hprev_t] + bc         (one GEMM per step, N = E lanes)
//                           gate blocks of Wc: r, u, hn (hidden part of the candidate), in (input part);
//                           pointwise: r, u = sigmoid, n = tanh(in + r hn), h' = (hprev - n) u + n,
//                           hprev_{t+1} = 0 where the episode ended (gru.rs:23-28); r, u, n, hn, h', hprev are kept per step
//   FVP tangent (R-operator along v): tG_t = Vc . [x_t ; hprev_t] + vbc + Wc[:, F:] . thprev_t  (two more GEMMs per step)
//   head + per-step algebra over all (t, e): logits, log-softmax, loss / KL / entropy, output cotangent dz (passes.cuh)
//   backward, t = T-1 .. 0  pointwise: dh' = act'(h') lw^T dz_t + carry  ->  D_t [4H x E] = (dpr, dpu, dpn r, dpn), carry = dh' u
//                           carry += W_hh^T [H x 3H] . D_t[0:3H]                               (one GEMM per step)
//   weight gradients        dWc [4H x (F + H + 1)] = sum_t D_t . [x_t ; hprev_t ; 1]^T          (ONE split-K GEMM over all (t, e))
//                           d lw, d lb [A x (H + 1)] = sum_t dz_t . [act(h'_t) ; 1]^T            (one more)
//
// The Hessian of mean KL(p0 || p_theta) at theta0 is J^T (diag p - p p^T) J for any network, so forward tangent +
// backward is the reference's double-backward Hessian-vector product (gru_update.cu header).
// Chain<Lstm, Linear> (a.cell = RL_CELL_LSTM) runs the same GEMMs with its own pointwise kernels: Wc [4H x (F + H)] holds the
// full [W_ih | W_hh] rows of all four gates i, f, g, o and bc = b_ih + b_hh; the gates kernel keeps i, f, g, o, h' per step and
// the cell state c before each step (plane CP); the backward pointwise carries (dh, dc) and emits D_t = the four gate
// pre-activation cotangents, after which carry += W_hh^T [H x 4H] . D_t; d b_ih = d b_hh.  The LSTM stays on the FP32 pipe.
//
// GEMMs: hand-written FP32 register-tiled kernels (128 x 128 x 8 tiles, 8 x 8 per thread, register-prefetched; the split-K
// one contracts over lanes with f64 flushes).  FP32, not tensor cores: the parity bar is 1e-5-class against f64 autograd, which bf16/tf32
// inputs miss; the bf16-piece tcgen05 form used by pass_tc.cuh is the next step (DESIGN.md section 9).
#include "passes.cuh"

#include <algorithm>

namespace {

constexpr int BN = 128, GEMM_THREADS = 256;

// ---------------------------------------------------------------------------------------------------------------------
// C [M x N] (+)= A [M x K] . B [K x N] (+ bias[m]);  A row-major (lda), B rows 0 .. K0-1 from B0 and K0 .. K-1 from B1 (both
// with row stride ldb = N's plane stride), C row-major (ldc).  N = lanes: every load along n is coalesced.
// (16 TM) x 128 tiles, K in chunks of 8, TM x 8 accumulators per thread (TM = 8: 64 FMAs per four LDS.128); the next chunk's
// global loads are in flight while the current one is multiplied.
// ---------------------------------------------------------------------------------------------------------------------
template <int TM>
__global__ void __launch_bounds__(GEMM_THREADS)
    gemm_nn_kernel(const float *__restrict__ A, int lda, const float *__restrict__ B0, const float *__restrict__ B1, int K0,
                   uint64_t ldb, float *__restrict__ C, uint64_t ldc, const float *__restrict__ bias, int accumulate, int M,
                   uint64_t N, int K, const int *skip_flag) {
    constexpr int TBM = 16 * TM, TBK = 8, AL = TBM * TBK / GEMM_THREADS;  // A values per thread and chunk: 4 (TM 8) or 2 (TM 4)
    if (skip_flag && *skip_flag) return;
    __shared__ __align__(16) float As[TBK][TBM + 4];
    __shared__ __align__(16) float Bs[TBK][BN];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;  // thread tile: rows ty * TM .. , cols tx * 4 .. + 3 and 64 + tx * 4 .. + 3
    const int m0 = blockIdx.y * TBM;
    const uint64_t n0 = (uint64_t)blockIdx.x * BN;
    float acc[TM][8];
#pragma unroll
    for (int i = 0; i < TM; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;
    float ra[AL], rb[4];
    const int bk = tid >> 5, bn = (tid & 31) * 4;  // B chunk: 8 rows x 128 lanes, one float4 per thread
    const bool vec_ok = (ldb & 3) == 0 && ((n0 + bn + 3) < N) && ((reinterpret_cast<uintptr_t>(B0) | reinterpret_cast<uintptr_t>(B1)) & 15) == 0;
    auto fetch = [&](int k0) {
#pragma unroll
        for (int i = 0; i < AL; ++i) {
            const int idx = tid + i * GEMM_THREADS, m = idx >> 3, k = idx & 7;
            ra[i] = (m0 + m < M && k0 + k < K) ? A[(size_t)(m0 + m) * lda + k0 + k] : 0.0f;
        }
        const int kk = k0 + bk;
        if (kk < K) {
            const float *src = kk < K0 ? B0 + (uint64_t)kk * ldb : B1 + (uint64_t)(kk - K0) * ldb;
            if (vec_ok) {
                const float4 v = *reinterpret_cast<const float4 *>(src + n0 + bn);
                rb[0] = v.x; rb[1] = v.y; rb[2] = v.z; rb[3] = v.w;
            } else {
#pragma unroll
                for (int j = 0; j < 4; ++j) rb[j] = (n0 + bn + j < N) ? src[n0 + bn + j] : 0.0f;
            }
        } else {
            rb[0] = rb[1] = rb[2] = rb[3] = 0.0f;
        }
    };
    fetch(0);
    for (int k0 = 0; k0 < K; k0 += TBK) {
#pragma unroll
        for (int i = 0; i < AL; ++i) {
            const int idx = tid + i * GEMM_THREADS;
            As[idx & 7][idx >> 3] = ra[i];
        }
        *reinterpret_cast<float4 *>(&Bs[bk][bn]) = make_float4(rb[0], rb[1], rb[2], rb[3]);
        __syncthreads();
        if (k0 + TBK < K) fetch(k0 + TBK);
#pragma unroll
        for (int k = 0; k < TBK; ++k) {
            float av[TM], bv[8];
#pragma unroll
            for (int i = 0; i < TM; i += 4) {
                const float4 a4 = *reinterpret_cast<const float4 *>(&As[k][ty * TM + i]);
                av[i] = a4.x; av[i + 1] = a4.y; av[i + 2] = a4.z; av[i + 3] = a4.w;
            }
            const float4 b0 = *reinterpret_cast<const float4 *>(&Bs[k][tx * 4]), b1 = *reinterpret_cast<const float4 *>(&Bs[k][64 + tx * 4]);
            bv[0] = b0.x; bv[1] = b0.y; bv[2] = b0.z; bv[3] = b0.w; bv[4] = b1.x; bv[5] = b1.y; bv[6] = b1.z; bv[7] = b1.w;
#pragma unroll
            for (int i = 0; i < TM; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(av[i], bv[j], acc[i][j]);
        }
        __syncthreads();
    }
#pragma unroll
    for (int i = 0; i < TM; ++i) {
        const int m = m0 + ty * TM + i;
        if (m >= M) continue;
        const float b = bias ? bias[m] : 0.0f;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const uint64_t n = n0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
            if (n >= N) continue;
            float *c = C + (uint64_t)m * ldc + n;
            *c = accumulate ? *c + (acc[i][j] + b) : acc[i][j] + b;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------------
// Split-K "A . B^T" over all (t, e):  part[s][m][n] = sum over the split's (t, e) of D[t][m][e] * In[t][n][e], where In's rows
// come from src0 (rows0 rows), src1 (rows1 rows) and a row of ones (n == rows0 + rows1).  128 x 64 output tiles, 16 lanes per
// unit, 8 x 4 per thread from lane-major shared tiles (three LDS.128 per 32 FMAs); f32 accumulators are flushed into f64
// every 128 units.
// ---------------------------------------------------------------------------------------------------------------------
constexpr int NT_BM = 128, NT_BN = 64, NT_BK = 16, NT_THREADS = 256;
__global__ void __launch_bounds__(NT_THREADS)
    gemm_nt_splitk_kernel(const float *__restrict__ D, int M, const float *__restrict__ src0, int rows0, const float *__restrict__ src1,
                          int rows1, uint64_t T, uint64_t E, double *__restrict__ part, int NB, int splits, const int *skip_flag) {
    if (skip_flag && *skip_flag) return;
    __shared__ __align__(16) float Ds[NT_BK][NT_BM + 4];
    __shared__ __align__(16) float Is[NT_BK][NT_BN + 4];
    const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;  // rows ty * 8 .. + 7, cols tx * 4 .. + 3
    const int m0 = blockIdx.y * NT_BM, n0 = blockIdx.x * NT_BN, s = blockIdx.z;
    const uint64_t upt = (E + NT_BK - 1) / NT_BK, units = T * upt;  // unit = 16 lanes of one step
    const uint64_t u_begin = units * (uint64_t)s / (uint64_t)splits, u_end = units * (uint64_t)(s + 1) / (uint64_t)splits;
    float acc[8][4];
    double tot[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) { acc[i][j] = 0.0f; tot[i][j] = 0.0; }
    const int NIN = rows0 + rows1;  // index of the ones row
    uint32_t since_flush = 0;
    float rd[8], ri[4];
    auto fetch = [&](uint64_t u) {
        const uint64_t t = u / upt, e0 = (u - t * upt) * NT_BK;
        // D tile [128 m][16 e]: 8 values per thread; In tile [64 n][16 e]: 4 per thread; e fastest
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int idx = tid + i * NT_THREADS, r = idx >> 4, k = idx & 15;
            const uint64_t e = e0 + k;
            const int m = m0 + r;
            rd[i] = (m < M && e < E) ? D[(t * M + m) * E + e] : 0.0f;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int idx = tid + i * NT_THREADS, r = idx >> 4, k = idx & 15;
            const uint64_t e = e0 + k;
            const int n = n0 + r;
            float v = 0.0f;
            if (e < E) {
                if (n < rows0) v = src0[(t * rows0 + n) * E + e];
                else if (n < NIN) v = src1[(t * rows1 + (n - rows0)) * E + e];
                else if (n == NIN) v = 1.0f;
            }
            ri[i] = v;
        }
    };
    if (u_begin < u_end) fetch(u_begin);
    for (uint64_t u = u_begin; u < u_end; ++u) {
#pragma unroll
        for (int i = 0; i < 8; ++i) {
            const int idx = tid + i * NT_THREADS;
            Ds[idx & 15][idx >> 4] = rd[i];
        }
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const int idx = tid + i * NT_THREADS;
            Is[idx & 15][idx >> 4] = ri[i];
        }
        __syncthreads();
        if (u + 1 < u_end) fetch(u + 1);
#pragma unroll
        for (int k = 0; k < NT_BK; ++k) {
            const float4 d0 = *reinterpret_cast<const float4 *>(&Ds[k][ty * 8]), d1 = *reinterpret_cast<const float4 *>(&Ds[k][ty * 8 + 4]);
            const float4 i4 = *reinterpret_cast<const float4 *>(&Is[k][tx * 4]);
            const float dv[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
            const float iv[4] = {i4.x, i4.y, i4.z, i4.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(dv[i], iv[j], acc[i][j]);
        }
        __syncthreads();
        if (++since_flush == 128) {
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 4; ++j) { tot[i][j] += (double)acc[i][j]; acc[i][j] = 0.0f; }
            since_flush = 0;
        }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int m = m0 + ty * 8 + i;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int n = n0 + tx * 4 + j;
            if (m < M && n < NB) part[((size_t)s * M + m) * NB + n] = tot[i][j] + (double)acc[i][j];
        }
    }
}

// sums[m][n] = sum_s part[s][m][n] in split order (deterministic)
__global__ void splitk_reduce_kernel(const double *__restrict__ part, int splits, int MN, double *__restrict__ sums, const int *skip_flag) {
    if (skip_flag && *skip_flag) return;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= MN) return;
    double s = 0.0;
    for (int k = 0; k < splits; ++k) s += part[(size_t)k * MN + i];
    sums[i] = s;
}

// ---------------------------------------------------------------------------------------------------------------------
// Combined weights of one parameter vector (theta or the FVP direction):
//   Wc [4H x KP], bc [4H]: gate blocks r, u, hn, in (see the header);  WhT [H x 3H]: W_hh^T with column blocks r, u, n.
// ---------------------------------------------------------------------------------------------------------------------
__global__ void big_comb_kernel(const float *__restrict__ th, int F, int H, float *__restrict__ Wc, float *__restrict__ bc,
                                float *__restrict__ WhT) {
    const int KP = F + H;
    const float *w_ih = th, *w_hh = th + (size_t)3 * H * F, *b_ih = w_hh + (size_t)3 * H * H, *b_hh = b_ih + 3 * H;
    const int total = 4 * H * KP;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < total; idx += gridDim.x * blockDim.x) {
        const int m = idx / KP, k = idx - m * KP, blk = m / H, j = m - blk * H;
        float v = 0.0f;
        if (blk < 2) v = k < F ? w_ih[(size_t)(blk * H + j) * F + k] : w_hh[(size_t)(blk * H + j) * H + (k - F)];
        else if (blk == 2) v = k < F ? 0.0f : w_hh[(size_t)(2 * H + j) * H + (k - F)];
        else v = k < F ? w_ih[(size_t)(2 * H + j) * F + k] : 0.0f;
        Wc[idx] = v;
    }
    for (int m = blockIdx.x * blockDim.x + threadIdx.x; m < 4 * H; m += gridDim.x * blockDim.x) {
        const int blk = m / H, j = m - blk * H;
        bc[m] = blk < 2 ? __fadd_rn(b_hh[blk * H + j], b_ih[blk * H + j]) : blk == 2 ? b_hh[2 * H + j] : b_ih[2 * H + j];
    }
    if (WhT)
        for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < 3 * H * H; idx += gridDim.x * blockDim.x) {
            const int k = idx / (3 * H), c = idx - k * 3 * H;  // WhT[k][c] = w_hh[c][k]
            WhT[idx] = w_hh[(size_t)c * H + k];
        }
}

// The LSTM's combined weights: Wc [4H x KP] = [W_ih | W_hh], bc = b_ih + b_hh, WhT [H x 4H] = W_hh^T
__global__ void lstm_comb_kernel(const float *__restrict__ th, int F, int H, float *__restrict__ Wc, float *__restrict__ bc,
                                 float *__restrict__ WhT) {
    const int KP = F + H;
    const float *w_ih = th, *w_hh = th + (size_t)4 * H * F, *b_ih = w_hh + (size_t)4 * H * H, *b_hh = b_ih + 4 * H;
    for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < 4 * H * KP; idx += gridDim.x * blockDim.x) {
        const int m = idx / KP, k = idx - m * KP;
        Wc[idx] = k < F ? w_ih[(size_t)m * F + k] : w_hh[(size_t)m * H + (k - F)];
    }
    for (int m = blockIdx.x * blockDim.x + threadIdx.x; m < 4 * H; m += gridDim.x * blockDim.x) bc[m] = __fadd_rn(b_ih[m], b_hh[m]);
    if (WhT)
        for (int idx = blockIdx.x * blockDim.x + threadIdx.x; idx < 4 * H * H; idx += gridDim.x * blockDim.x) {
            const int k = idx / (4 * H), c = idx - k * 4 * H;  // WhT[k][c] = w_hh[c][k]
            WhT[idx] = w_hh[(size_t)c * H + k];
        }
}

__global__ void big_zero_kernel(float *p, uint64_t n, const int *skip_flag) {
    if (skip_flag && *skip_flag) return;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) p[i] = 0.0f;
}

struct BigPlanes {
    float *G, *tG;                        // [4H][E] of the current step
    float *R, *U, *N, *HN, *HNEW, *AV;    // [T][H][E]; an LSTM keeps its gates i, f, g, o in R, U, N, HN
    float *THNEW;                         // [T][H][E] (FVP)
    float *thp, *dh;                      // [H][E]
    float *D;                             // [T][4H][E]
    float *CP;                            // [T][H][E] LSTM: cell state before each step
    float *tcp, *dc;                      // [H][E] LSTM: tangent of c (FVP), cell-state carry (backward)
};

// gates of step t from G (biases included) and hprev = hbuf[t]
__global__ void big_gates_kernel(const float *__restrict__ G, const float *__restrict__ hprev, const uint8_t *__restrict__ succ_t,
                                 float *__restrict__ R, float *__restrict__ U, float *__restrict__ Nn, float *__restrict__ HN,
                                 float *__restrict__ HNEW, float *__restrict__ hnext, int H, uint64_t E, const int *skip_flag) {
    if (skip_flag && *skip_flag) return;
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (uint64_t)H * E) return;
    const uint64_t j = i / E, e = i - j * E, HE = (uint64_t)H * E;
    const float r = sigm(G[i]), u = sigm(G[HE + i]), hn = G[2 * HE + i], in = G[3 * HE + i];
    const float n = tanhf(__fadd_rn(in, __fmul_rn(hn, r)));
    const float hp = hprev[i];
    const float hnew = __fadd_rn(__fmul_rn(__fsub_rn(hp, n), u), n);
    R[i] = r; U[i] = u; Nn[i] = n; HN[i] = hn; HNEW[i] = hnew;
    if (hnext) hnext[i] = succ_t[e] != RL_CONTINUE ? 0.0f : hnew;  // a new episode starts from zeros; padding stays zero too
}

// lstm_cell of step t from G (biases included) and cprev: gates, h' = o tanh(c'), c' = f cprev + i g (to cout when given); the
// next step's (h, c) are zero where the episode ended
__global__ void lstm_gates_kernel(const float *__restrict__ G, const float *__restrict__ cprev, const uint8_t *__restrict__ succ_t,
                                  float *__restrict__ I, float *__restrict__ Fg, float *__restrict__ Gg, float *__restrict__ O,
                                  float *__restrict__ HNEW, float *__restrict__ cout, float *__restrict__ hnext, float *__restrict__ cnext,
                                  int H, uint64_t E, const int *skip_flag) {
    if (skip_flag && *skip_flag) return;
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (uint64_t)H * E) return;
    const uint64_t j = i / E, e = i - j * E, HE = (uint64_t)H * E;
    const float ig = sigm(G[i]), fg = sigm(G[HE + i]), gg = tanhf(G[2 * HE + i]), og = sigm(G[3 * HE + i]);
    const float c = __fadd_rn(__fmul_rn(fg, cprev[i]), __fmul_rn(ig, gg));
    const float hnew = __fmul_rn(og, tanhf(c));
    I[i] = ig; Fg[i] = fg; Gg[i] = gg; O[i] = og; HNEW[i] = hnew;
    if (cout) cout[i] = c;
    const bool done = succ_t[e] != RL_CONTINUE;
    if (hnext) hnext[i] = done ? 0.0f : hnew;
    if (cnext) cnext[i] = done ? 0.0f : c;
}

// LSTM tangents along v: tG = V [x; hprev] + vb + W_hh thprev (all four gate blocks); carries (thp, tcp) cut at episode ends
__global__ void lstm_gates_tan_kernel(const float *__restrict__ tG, const float *__restrict__ I, const float *__restrict__ Fg,
                                      const float *__restrict__ Gg, const float *__restrict__ O, const float *__restrict__ cprev,
                                      float *__restrict__ thp, float *__restrict__ tcp, float *__restrict__ THNEW,
                                      const uint8_t *__restrict__ succ_t, int H, uint64_t E, const int *skip_flag) {
    if (skip_flag && *skip_flag) return;
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (uint64_t)H * E) return;
    const uint64_t j = i / E, e = i - j * E, HE = (uint64_t)H * E;
    const float ig = I[i], fg = Fg[i], gg = Gg[i], og = O[i], cp = cprev[i];
    const float tc = tanhf(__fadd_rn(__fmul_rn(fg, cp), __fmul_rn(ig, gg)));
    const float id = ig * (1.0f - ig) * tG[i], fd = fg * (1.0f - fg) * tG[HE + i];
    const float gd = (1.0f - gg * gg) * tG[2 * HE + i], od = og * (1.0f - og) * tG[3 * HE + i];
    const float tcn = fd * cp + fg * tcp[i] + id * gg + ig * gd;
    const float thn = od * tc + og * (1.0f - tc * tc) * tcn;
    THNEW[i] = thn;
    const bool done = succ_t[e] != RL_CONTINUE;
    thp[i] = done ? 0.0f : thn;
    tcp[i] = done ? 0.0f : tcn;
}

// tangent of the gates along v (R-operator): tG = V [x; hprev] + vb + W[:, F:] thprev
__global__ void big_gates_tan_kernel(const float *__restrict__ tG, const float *__restrict__ R, const float *__restrict__ U,
                                     const float *__restrict__ Nn, const float *__restrict__ HN, const float *__restrict__ hprev,
                                     float *__restrict__ thp, float *__restrict__ THNEW, const uint8_t *__restrict__ succ_t, int H,
                                     uint64_t E, const int *skip_flag) {
    if (skip_flag && *skip_flag) return;
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (uint64_t)H * E) return;
    const uint64_t j = i / E, e = i - j * E, HE = (uint64_t)H * E;
    const float r = R[i], u = U[i], n = Nn[i], hn = HN[i];
    const float rd = r * (1.0f - r) * tG[i];
    const float ud = u * (1.0f - u) * tG[HE + i];
    const float nd = (1.0f - n * n) * (tG[3 * HE + i] + rd * hn + r * tG[2 * HE + i]);
    const float thnew = ud * (hprev[i] - n) + u * thp[i] + (1.0f - u) * nd;
    THNEW[i] = thnew;
    thp[i] = succ_t[e] != RL_CONTINUE ? 0.0f : thnew;
}

// Linear head + the per-step loss algebra (passes.cuh) over all (t, e); one partial of the four scalar sums per block
constexpr int HEAD_THREADS = 128, HEAD_MAXA_ALL = 32;
// HEAD_MAXA = the compile-time bound of the per-thread arrays over the outputs (logits, probabilities, cotangent): 16 keeps
// them in registers for the module sizes of the experiments (2 .. 10 arms); 32 serves the rest through local memory
template <int MODE, int HEAD_MAXA>
__global__ void __launch_bounds__(HEAD_THREADS) big_head_kernel(rl_seq_pass_args a, const float *__restrict__ HNEW,
                                                                const float *__restrict__ THNEW, double *__restrict__ scal_part) {
    using M = PassMode<MODE>;
    constexpr bool FVP = M::FVP;
    if (a.skip_flag && *a.skip_flag) return;
    extern __shared__ float hsm[];  // lw [A][H], lb [A], (FVP) vlw, vlb
    const int H = a.H, A = a.A, F = a.F, NG = rl_cell_gates(a.cell);
    const int o_lw = NG * H * F + NG * H * H + 2 * NG * H;
    float *lw = hsm, *lb = lw + A * H, *vlw = lb + A, *vlb = vlw + A * H;
    for (int i = threadIdx.x; i < A * H + A; i += blockDim.x) {
        lw[i] = a.theta[o_lw + i];
        if (FVP) vlw[i] = a.vec[o_lw + i];  // (vlw and vlb are contiguous like lw and lb)
    }
    __syncthreads();
    const uint64_t E = a.E, TE = a.T * E;
    const uint64_t idx = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    double s_loss = 0.0, s_kl = 0.0, s_ent = 0.0, s_cnt = 0.0;
    if (idx < TE) {
        const uint64_t t = idx / E, e = idx - t * E;
        const uint8_t sc = a.succ[idx];
        float dz[HEAD_MAXA];
#pragma unroll
        for (int k = 0; k < HEAD_MAXA; ++k) dz[k] = 0.0f;
        if (sc != RL_PAD) {
            float z[HEAD_MAXA], zd[HEAD_MAXA];
#pragma unroll
            for (int k = 0; k < HEAD_MAXA; ++k) {
                z[k] = k < A ? lb[k] : 0.0f;
                zd[k] = (FVP && k < A) ? vlb[k] : 0.0f;
            }
            for (int j = 0; j < H; ++j) {
                const float hn = HNEW[(t * H + j) * E + e];
                const float av = rl_activate(a.act, hn);
                const float gd = FVP ? act_grad(a.act, hn, av) * THNEW[(t * H + j) * E + e] : 0.0f;
#pragma unroll
                for (int k = 0; k < HEAD_MAXA; ++k)
                    if (k < A) {
                        z[k] = fmaf(lw[k * H + j], av, z[k]);
                        if (FVP) zd[k] = fmaf(vlw[k * H + j], av, fmaf(lw[k * H + j], gd, zd[k]));
                    }
            }
            float lp[HEAD_MAXA];
            const SampleLoss ls = sample_loss<MODE, HEAD_MAXA>(z, zd, A, M::USES_ACT ? (int)a.action[idx] : 0, M::USES_ADV ? a.adv[idx] : 0.0f,
                                                               M::USES_TARGET ? a.target[idx] : 0.0f, make_float2(a.clip_lo, a.clip_hi),
                                                               [&](int k) { return a.logp0[(t * A + k) * E + e]; }, lp, dz);
            if (MODE == RL_PASS_STATS) {
#pragma unroll
                for (int k = 0; k < HEAD_MAXA; ++k)
                    if (k < A) a.logp0[(t * A + k) * E + e] = lp[k];
            }
            s_cnt = 1.0; s_loss = (double)ls.loss; s_kl = (double)ls.kl; s_ent = (double)ls.entropy;
        }
        if (M::BACKWARD) {
#pragma unroll
            for (int k = 0; k < HEAD_MAXA; ++k)
                if (k < A) a.dzbuf[(t * A + k) * E + e] = dz[k];  // zero on padding
        }
    }
    // block partial of the scalar sums (fixed order: warp shuffle tree, then warps in order)
    __shared__ double red[HEAD_THREADS / 32][4];
    auto wsum = [](double v) {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        return v;
    };
    const double v0 = wsum(s_loss), v1 = wsum(s_kl), v2 = wsum(s_ent), v3 = wsum(s_cnt);
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) { red[warp][0] = v0; red[warp][1] = v1; red[warp][2] = v2; red[warp][3] = v3; }
    __syncthreads();
    if (threadIdx.x < 4) {
        double s = 0.0;
        for (int w = 0; w < HEAD_THREADS / 32; ++w) s += red[w][threadIdx.x];
        scal_part[(size_t)blockIdx.x * 4 + threadIdx.x] = s;
    }
}

// backward pointwise of step t: D_t, AV_t, and the carry dh := dh' u  (the GEMM adds W_hh^T D_t[0:3H] afterwards)
__global__ void big_bwd_kernel(const float *__restrict__ dz_t, const float *__restrict__ theta, int o_lw, int act,
                               const float *__restrict__ R, const float *__restrict__ U, const float *__restrict__ Nn,
                               const float *__restrict__ HN, const float *__restrict__ HNEW, const float *__restrict__ hprev,
                               const uint8_t *__restrict__ succ_t, float *__restrict__ dh, float *__restrict__ D, float *__restrict__ AV,
                               int H, int A, uint64_t E, const int *skip_flag) {
    if (skip_flag && *skip_flag) return;
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (uint64_t)H * E) return;
    const uint64_t j = i / E, e = i - j * E, HE = (uint64_t)H * E;
    const uint8_t sc = succ_t[e];
    if (sc == RL_PAD) {
        D[i] = 0.0f; D[HE + i] = 0.0f; D[2 * HE + i] = 0.0f; D[3 * HE + i] = 0.0f;
        AV[i] = 0.0f;
        dh[i] = 0.0f;
        return;
    }
    const float *lw = theta + o_lw;
    float da = 0.0f;
    for (int k = 0; k < A; ++k) da = fmaf(lw[k * H + j], dz_t[(uint64_t)k * E + e], da);
    const float hnew = HNEW[i], av = rl_activate(act, hnew);
    AV[i] = av;
    const float carry = sc != RL_CONTINUE ? 0.0f : dh[i];  // last step of its episode: nothing flows back from t + 1
    const float dhn = fmaf(act_grad(act, hnew, av), da, carry);
    const float r = R[i], u = U[i], n = Nn[i], hn = HN[i], hp = hprev[i];
    // h' = u h + (1 - u) n
    const float du = dhn * (hp - n), dn = dhn * (1.0f - u);
    const float dpn = dn * (1.0f - n * n);
    const float dr = dpn * hn;
    const float dpu = du * u * (1.0f - u);
    const float dpr = dr * r * (1.0f - r);
    D[i] = dpr; D[HE + i] = dpu; D[2 * HE + i] = dpn * r; D[3 * HE + i] = dpn;
    dh[i] = dhn * u;
}

// LSTM backward pointwise of step t: D_t = (di, df, dg, do), AV_t, the cell-state carry dc := dc' f, and dh := 0 for the GEMM
// that adds W_hh^T D_t
__global__ void lstm_bwd_kernel(const float *__restrict__ dz_t, const float *__restrict__ theta, int o_lw, int act,
                                const float *__restrict__ I, const float *__restrict__ Fg, const float *__restrict__ Gg,
                                const float *__restrict__ O, const float *__restrict__ HNEW, const float *__restrict__ cprev,
                                const uint8_t *__restrict__ succ_t, float *__restrict__ dh, float *__restrict__ dc, float *__restrict__ D,
                                float *__restrict__ AV, int H, int A, uint64_t E, const int *skip_flag) {
    if (skip_flag && *skip_flag) return;
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (uint64_t)H * E) return;
    const uint64_t j = i / E, e = i - j * E, HE = (uint64_t)H * E;
    const uint8_t sc = succ_t[e];
    if (sc == RL_PAD) {
        D[i] = 0.0f; D[HE + i] = 0.0f; D[2 * HE + i] = 0.0f; D[3 * HE + i] = 0.0f;
        AV[i] = 0.0f;
        dh[i] = 0.0f;
        dc[i] = 0.0f;
        return;
    }
    const float *lw = theta + o_lw;
    float da = 0.0f;
    for (int k = 0; k < A; ++k) da = fmaf(lw[k * H + j], dz_t[(uint64_t)k * E + e], da);
    const float hnew = HNEW[i], av = rl_activate(act, hnew);
    AV[i] = av;
    const bool last = sc != RL_CONTINUE;  // last step of its episode: nothing flows back from t + 1
    const float dhn = fmaf(act_grad(act, hnew, av), da, last ? 0.0f : dh[i]);
    const float ig = I[i], fg = Fg[i], gg = Gg[i], og = O[i], cp = cprev[i];
    const float tc = tanhf(__fadd_rn(__fmul_rn(fg, cp), __fmul_rn(ig, gg)));
    const float dcn = (last ? 0.0f : dc[i]) + dhn * og * (1.0f - tc * tc);
    D[i] = dcn * gg * ig * (1.0f - ig);
    D[HE + i] = dcn * cp * fg * (1.0f - fg);
    D[2 * HE + i] = dcn * ig * (1.0f - gg * gg);
    D[3 * HE + i] = dhn * tc * og * (1.0f - og);
    dc[i] = dcn * fg;
    dh[i] = 0.0f;
}

// the partial row: parameter order w_ih, w_hh, b_ih, b_hh, lw, lb, then loss, kl, entropy, count.  An LSTM's rows of dWc are
// its parameter rows in order (Wc = [W_ih | W_hh]), and its two bias gradients are the same column.
template <int CELL>
__device__ __forceinline__ void assemble(const double *__restrict__ dWc, const double *__restrict__ dHead, const double *__restrict__ scal_part,
                                         int nscal, int F, int H, int A, int backward, double *__restrict__ row, const int *skip_flag) {
    if (skip_flag && *skip_flag) return;
    const int KP = F + H, NB = KP + 1, NH = H + 1;
    constexpr int NG = rl_cell_gates(CELL);
    const int o_whh = NG * H * F, o_bih = o_whh + NG * H * H, o_bhh = o_bih + NG * H, o_lw = o_bhh + NG * H, o_lb = o_lw + A * H, P = o_lb + A;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < P; i += gridDim.x * blockDim.x) {
        double v = 0.0;
        if (CELL == RL_CELL_LSTM && backward && i < o_lw) {
            if (i < o_whh) {
                const int row_ = i / F, f = i - row_ * F;
                v = dWc[(size_t)row_ * NB + f];
            } else if (i < o_bih) {
                const int q = i - o_whh, row_ = q / H, k = q - row_ * H;
                v = dWc[(size_t)row_ * NB + F + k];
            } else {
                v = dWc[(size_t)((i - o_bih) % (4 * H)) * NB + KP];
            }
        } else if (backward) {
            if (i < o_whh) {  // w_ih[g H + j][f]: gates r, u from blocks 0, 1; n from block 3 (input part)
                const int row_ = i / F, f = i - row_ * F, g = row_ / H, j = row_ - g * H, blk = g < 2 ? g : 3;
                v = dWc[(size_t)(blk * H + j) * NB + f];
            } else if (i < o_bih) {  // w_hh[g H + j][k]: n from block 2 (hidden part)
                const int q = i - o_whh, row_ = q / H, k = q - row_ * H, g = row_ / H, j = row_ - g * H;
                v = dWc[(size_t)(g * H + j) * NB + F + k];
            } else if (i < o_bhh) {
                const int row_ = i - o_bih, g = row_ / H, j = row_ - g * H, blk = g < 2 ? g : 3;
                v = dWc[(size_t)(blk * H + j) * NB + KP];
            } else if (i < o_lw) {
                const int row_ = i - o_bhh, g = row_ / H, j = row_ - g * H;
                v = dWc[(size_t)(g * H + j) * NB + KP];
            } else if (i < o_lb) {
                const int q = i - o_lw, k = q / H, j = q - k * H;
                v = dHead[(size_t)k * NH + j];
            } else {
                v = dHead[(size_t)(i - o_lb) * NH + H];
            }
        }
        row[i] = v;
    }
    if (blockIdx.x == 0) {
        // the four scalar sums over the head kernel's block partials: 64 strided chains per scalar, then a fixed-order tree
        __shared__ double red[4][64];
        const int sc = threadIdx.x >> 6, ln = threadIdx.x & 63;  // 256 threads = 4 scalars x 64 chains
        double s = 0.0;
        for (int b = ln; b < nscal; b += 64) s += scal_part[(size_t)b * 4 + sc];
        red[sc][ln] = s;
        __syncthreads();
        for (int w = 32; w > 0; w >>= 1) {
            if (ln < w) red[sc][ln] += red[sc][ln + w];
            __syncthreads();
        }
        if (ln == 0) row[P + sc] = red[sc][0];
    }
}

__global__ void big_assemble_kernel(const double *__restrict__ dWc, const double *__restrict__ dHead, const double *__restrict__ scal_part,
                                    int nscal, int F, int H, int A, int backward, double *__restrict__ row, const int *skip_flag) {
    assemble<RL_CELL_GRU>(dWc, dHead, scal_part, nscal, F, H, A, backward, row, skip_flag);
}

__global__ void lstm_assemble_kernel(const double *__restrict__ dWc, const double *__restrict__ dHead, const double *__restrict__ scal_part,
                                     int nscal, int F, int H, int A, int backward, double *__restrict__ row, const int *skip_flag) {
    assemble<RL_CELL_LSTM>(dWc, dHead, scal_part, nscal, F, H, A, backward, row, skip_flag);
}

// outputs of the Linear head for one step: out[k][e] = lb[k] + sum_j lw[k][j] act(hnew[j][e]); zero where `only` is given and
// the step's successor code differs from it (out_next: only interrupted steps), and on padding
__global__ void __launch_bounds__(128) big_head_out_kernel(const float *__restrict__ theta, int o_lw, int act, const float *__restrict__ HNEW,
                                                          const uint8_t *__restrict__ succ_t, int only, float *__restrict__ out_t, int H,
                                                          int A, uint64_t E) {
    extern __shared__ float hsm2[];  // lw [A][H], lb [A]
    for (int i = threadIdx.x; i < A * H + A; i += blockDim.x) hsm2[i] = theta[o_lw + i];
    __syncthreads();
    const uint64_t e = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= E) return;
    const uint8_t sc = succ_t[e];
    const bool live = sc != RL_PAD && (only < 0 || sc == only);
    constexpr int HEAD_MAXA = HEAD_MAXA_ALL;
    float z[HEAD_MAXA];
#pragma unroll
    for (int k = 0; k < HEAD_MAXA; ++k) z[k] = k < A ? hsm2[A * H + k] : 0.0f;
    if (live)
        for (int j = 0; j < H; ++j) {
            const float av = rl_activate(act, HNEW[(uint64_t)j * E + e]);
#pragma unroll
            for (int k = 0; k < HEAD_MAXA; ++k)
                if (k < A) z[k] = fmaf(hsm2[k * H + j], av, z[k]);
        }
#pragma unroll
    for (int k = 0; k < HEAD_MAXA; ++k)
        if (k < A) out_t[(uint64_t)k * E + e] = live ? z[k] : 0.0f;
}

#include "gru_big_tc.cuh"

// RL_SEQ_TC=0 keeps the per-step GEMMs on the FP32 pipe (cross-check / measurements)
bool seq_tc_enabled() {
    static int v = -1;
    if (v < 0) {
        const char *e = getenv("RL_SEQ_TC");
        v = (e && e[0] == '0') ? 0 : 1;
    }
    return v == 1;
}

template <int N, int EPI>
rl_status launch_tc(rl_ctx *ctx, const bt::BtArgs &a_in) {
    bt::BtArgs a = a_in;
    static long long *dbg = nullptr;
    static int dbg_left = getenv("RL_SEQ_TC_DEBUG") ? 3 : 0;
    if (dbg_left > 0) {
        if (!dbg) cudaMallocManaged(&dbg, 64);
        cudaDeviceSynchronize();
        a.dbg = dbg;
    }
    static bool configured = false;
    if (!configured) {
        RL_CUDA(ctx, cudaFuncSetAttribute(bt::big_gemm_tc_kernel<N, EPI>, cudaFuncAttributeMaxDynamicSharedMemorySize, bt::bt_smem(N)));
        configured = true;
    }
    RL_LAUNCH(ctx, (bt::big_gemm_tc_kernel<N, EPI>), (unsigned)rl_div_up(a.E, bt::BT_LANES), bt::BT_THREADS, bt::bt_smem(N), a);
    if (dbg_left > 0) {
        cudaDeviceSynchronize();
        fprintf(stderr, "big_gemm_tc<%d,%d> nsteps %d: setup %lld clk, steps %lld clk, epilogue %lld clk\n", N, EPI, a.nsteps, dbg[0], dbg[1], dbg[2]);
        --dbg_left;
    }
    return RL_OK;
}

template <int MODE>
rl_status launch_head(rl_ctx *ctx, const rl_seq_pass_args &a, const BigPlanes &pl, double *scal_part, int blocks) {
    const size_t smem = (size_t)2 * (a.A * a.H + a.A) * sizeof(float);
    if (a.A <= 16) RL_LAUNCH(ctx, (big_head_kernel<MODE, 16>), blocks, HEAD_THREADS, smem, a, pl.HNEW, pl.THNEW, scal_part);
    else RL_LAUNCH(ctx, (big_head_kernel<MODE, HEAD_MAXA_ALL>), blocks, HEAD_THREADS, smem, a, pl.HNEW, pl.THNEW, scal_part);
    return RL_OK;
}

rl_status gemm_nn(rl_ctx *ctx, const float *A, int lda, const float *B0, const float *B1, int K0, uint64_t ldb, float *C, uint64_t ldc,
                  const float *bias, int accumulate, int M, uint64_t N, int K, const int *skip_flag) {
    // 128-row tiles while they give at least two CTAs per SM, else 64-row tiles (the H-row carry GEMM of the backward sweep)
    const uint64_t ctas128 = rl_div_up(N, BN) * rl_div_up(M, 128);
    if (M >= 128 && ctas128 >= (uint64_t)2 * ctx->sm_count) {
        dim3 grid((unsigned)rl_div_up(N, BN), (unsigned)rl_div_up(M, 128));
        RL_LAUNCH(ctx, gemm_nn_kernel<8>, grid, GEMM_THREADS, 0, A, lda, B0, B1, K0, ldb, C, ldc, bias, accumulate, M, N, K, skip_flag);
    } else {
        dim3 grid((unsigned)rl_div_up(N, BN), (unsigned)rl_div_up(M, 64));
        RL_LAUNCH(ctx, gemm_nn_kernel<4>, grid, GEMM_THREADS, 0, A, lda, B0, B1, K0, ldb, C, ldc, bias, accumulate, M, N, K, skip_flag);
    }
    return RL_OK;
}

}  // namespace

bool rl_seq_big_supports(int F, int H, int A) { return F >= 1 && F <= 64 && H >= 1 && H <= 128 && A >= 1 && A <= HEAD_MAXA_ALL; }

// One pass through the GEMM formulation; writes ONE partial row of P + 4 doubles at a.partials.
rl_status rl_seq_big_pass_launch(rl_ctx *ctx, int mode, const rl_seq_pass_args &a) {
    const int F = a.F, H = a.H, A = a.A, KP = F + H, NB = KP + 1, NH = H + 1;
    const uint64_t T = a.T, E = a.E, HE = (uint64_t)H * E, TE = T * E;
    const bool fvp = mode == RL_PASS_FVP;
    const bool backward = pass_backward(mode);
    const bool lstm = a.cell == RL_CELL_LSTM;
    const int NG = rl_cell_gates(a.cell);
    const int *skip = a.skip_flag;
    // ---- scratch (second context scratch: the plan and hbuf / dzbuf / logp0 live in the first) ----
    const int splits = 32;
    const int head_blocks = (int)rl_div_up(TE, HEAD_THREADS);
    auto al = [](size_t b) { return (b + 255) / 256 * 256; };
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += al(bytes); return o; };
    const size_t o_Wc = take((size_t)4 * H * KP * 4), o_bc = take((size_t)4 * H * 4), o_WhT = take((size_t)NG * H * H * 4);
    const size_t o_Vc = take((size_t)4 * H * KP * 4), o_vbc = take((size_t)4 * H * 4);
    const size_t o_G = take(4 * HE * 4), o_tG = take(fvp ? 4 * HE * 4 : 0), o_thp = take(fvp ? HE * 4 : 0), o_dh = take(backward ? HE * 4 : 0);
    const size_t plane = T * HE * 4;
    const size_t o_R = take(plane), o_U = take(plane), o_N = take(plane), o_HN = take(plane), o_HNEW = take(plane);
    const size_t o_AV = take(backward ? plane : 0), o_TH = take(fvp ? plane : 0), o_D = take(backward ? 4 * plane : 0);
    const size_t o_partW = take(backward ? (size_t)splits * 4 * H * NB * 8 : 0), o_partH = take(backward ? (size_t)splits * A * NH * 8 : 0);
    const size_t o_dWc = take((size_t)4 * H * NB * 8), o_dHead = take((size_t)A * NH * 8), o_scal = take((size_t)head_blocks * 4 * 8);
    const size_t o_CP = take(lstm ? plane : 0), o_tcp = take(lstm && fvp ? HE * 4 : 0), o_dc = take(lstm && backward ? HE * 4 : 0);
    // tensor-core form of the per-step GEMMs (gru_big_tc.cuh, GRU cells only): weight pieces of the three matrices
    const bool use_tc = H == 128 && seq_tc_enabled() && !lstm;
    const int stW = (KP + 15) / 16, stT = (KP + H + 15) / 16, stB = (3 * H + 15) / 16;
    const size_t o_wpW = take(use_tc ? (size_t)stW * bt::bt_b_stage(512) : 0), o_wpT = take(use_tc && fvp ? (size_t)stT * bt::bt_b_stage(512) : 0);
    const size_t o_wpB = take(use_tc && backward ? (size_t)stB * bt::bt_b_stage(128) : 0);
    // weight gradients on the tensor cores: one split per SM and M half, f32 slabs drained every NT_DRAIN steps
    const bool nt_tc = use_tc && backward && KP + 1 <= bt::NT_ROWS_B;
    const int nt_splits = ctx->sm_count / 2 > 0 ? ctx->sm_count / 2 : 1;
    const uint64_t nt_units = T * ((E + 15) / 16);
    const int nt_nd = (int)rl_div_up(rl_div_up(nt_units, (uint64_t)nt_splits) + 1, (uint64_t)bt::NT_DRAIN);
    const size_t nt_part_bytes = (size_t)nt_splits * nt_nd * 2 * bt::NT_ROWS_A * bt::NT_ROWS_B * sizeof(float);
    const size_t o_ntpart = take(nt_tc ? nt_part_bytes : 0);
    char *base;
    RL_TRY(rl_ctx_scratch2(ctx, off + 256, (void **)&base));
    uint16_t *wpW = (uint16_t *)(base + o_wpW), *wpT = (uint16_t *)(base + o_wpT), *wpB = (uint16_t *)(base + o_wpB);
    float *Wc = (float *)(base + o_Wc), *bc = (float *)(base + o_bc), *WhT = (float *)(base + o_WhT);
    float *Vc = (float *)(base + o_Vc), *vbc = (float *)(base + o_vbc);
    BigPlanes pl{};
    pl.G = (float *)(base + o_G); pl.tG = (float *)(base + o_tG); pl.thp = (float *)(base + o_thp); pl.dh = (float *)(base + o_dh);
    pl.R = (float *)(base + o_R); pl.U = (float *)(base + o_U); pl.N = (float *)(base + o_N); pl.HN = (float *)(base + o_HN);
    pl.HNEW = (float *)(base + o_HNEW); pl.AV = (float *)(base + o_AV); pl.THNEW = (float *)(base + o_TH); pl.D = (float *)(base + o_D);
    pl.CP = (float *)(base + o_CP); pl.tcp = (float *)(base + o_tcp); pl.dc = (float *)(base + o_dc);
    double *partW = (double *)(base + o_partW), *partH = (double *)(base + o_partH), *dWc = (double *)(base + o_dWc),
           *dHead = (double *)(base + o_dHead), *scal_part = (double *)(base + o_scal);
    const unsigned pw_grid = (unsigned)rl_div_up(HE, 256);
    if (use_tc) {
        // The tensor-core GEMMs take 184 .. 196 KB of shared memory; the pointwise kernels launched between them take none.
        // Asking for the same (maximum) carve-out everywhere keeps the SMs from re-partitioning L1 / shared memory at every
        // launch boundary of the per-step sequences.
        static bool carved = false;
        if (!carved) {
            cudaFuncSetAttribute(big_bwd_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
            cudaFuncSetAttribute(big_zero_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
            cudaFuncSetAttribute(big_head_out_kernel, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
            carved = true;
        }
    }

    // ---- forward (and the tangent along a.vec) ----
    auto comb = lstm ? lstm_comb_kernel : big_comb_kernel;
    RL_LAUNCH(ctx, comb, 64, 256, 0, a.theta, F, H, Wc, bc, WhT);
    if (fvp) RL_LAUNCH(ctx, comb, 64, 256, 0, a.vec, F, H, Vc, vbc, (float *)nullptr);
    if (use_tc) {
        RL_LAUNCH(ctx, bt::big_pieces_kernel, 128, 256, 0, Wc, KP, KP, (const float *)nullptr, 0, 0, 4 * H, stW, wpW);
        if (fvp) RL_LAUNCH(ctx, bt::big_pieces_kernel, 128, 256, 0, Vc, KP, KP, Wc + F, KP, H, 4 * H, stT, wpT);
        if (backward) RL_LAUNCH(ctx, bt::big_pieces_kernel, 128, 256, 0, WhT, 3 * H, 3 * H, (const float *)nullptr, 0, 0, H, stB, wpB);
    }
    RL_LAUNCH(ctx, big_zero_kernel, 256, 256, 0, a.hbuf, HE, skip);  // SeqIterative::initial_state (gru.rs:23-28)
    if (fvp) RL_LAUNCH(ctx, big_zero_kernel, 256, 256, 0, pl.thp, HE, skip);
    if (lstm) RL_LAUNCH(ctx, big_zero_kernel, 256, 256, 0, pl.CP, HE, skip);
    if (lstm && fvp) RL_LAUNCH(ctx, big_zero_kernel, 256, 256, 0, pl.tcp, HE, skip);
    for (uint64_t t = 0; t < T; ++t) {
        const float *x_t = a.obs + t * (uint64_t)F * E, *hp_t = a.hbuf + t * HE;
        const uint8_t *succ_t = a.succ + t * E;
        if (use_tc) {
            bt::BtArgs g{};
            g.src0 = x_t; g.src1 = hp_t; g.src2 = hp_t; g.k0 = F; g.k1 = KP; g.K = KP; g.nsteps = stW; g.wp = wpW; g.E = E; g.bias = bc;
            g.succ_t = succ_t; g.R = pl.R + t * HE; g.U = pl.U + t * HE; g.Nn = pl.N + t * HE; g.HN = pl.HN + t * HE; g.HNEW = pl.HNEW + t * HE;
            g.hnext = t + 1 < T ? a.hbuf + (t + 1) * HE : nullptr; g.skip_flag = skip;
            RL_TRY((launch_tc<512, bt::EPI_GATES>(ctx, g)));
            if (fvp) {
                g.src2 = pl.thp; g.K = KP + H; g.nsteps = stT; g.wp = wpT; g.bias = vbc; g.THNEW = pl.THNEW + t * HE; g.thp = pl.thp;
                RL_TRY((launch_tc<512, bt::EPI_TAN>(ctx, g)));
            }
            continue;
        }
        RL_TRY(gemm_nn(ctx, Wc, KP, x_t, hp_t, F, E, pl.G, E, bc, 0, 4 * H, E, KP, skip));
        if (lstm)
            RL_LAUNCH(ctx, lstm_gates_kernel, pw_grid, 256, 0, pl.G, pl.CP + t * HE, succ_t, pl.R + t * HE, pl.U + t * HE, pl.N + t * HE,
                      pl.HN + t * HE, pl.HNEW + t * HE, (float *)nullptr, t + 1 < T ? a.hbuf + (t + 1) * HE : (float *)nullptr,
                      t + 1 < T ? pl.CP + (t + 1) * HE : (float *)nullptr, H, E, skip);
        else
            RL_LAUNCH(ctx, big_gates_kernel, pw_grid, 256, 0, pl.G, hp_t, succ_t, pl.R + t * HE, pl.U + t * HE, pl.N + t * HE, pl.HN + t * HE,
                      pl.HNEW + t * HE, t + 1 < T ? a.hbuf + (t + 1) * HE : (float *)nullptr, H, E, skip);
        if (fvp) {
            RL_TRY(gemm_nn(ctx, Vc, KP, x_t, hp_t, F, E, pl.tG, E, vbc, 0, 4 * H, E, KP, skip));
            RL_TRY(gemm_nn(ctx, Wc + F, KP, pl.thp, pl.thp, H, E, pl.tG, E, nullptr, 1, 4 * H, E, H, skip));
            if (lstm)
                RL_LAUNCH(ctx, lstm_gates_tan_kernel, pw_grid, 256, 0, pl.tG, pl.R + t * HE, pl.U + t * HE, pl.N + t * HE, pl.HN + t * HE,
                          pl.CP + t * HE, pl.thp, pl.tcp, pl.THNEW + t * HE, succ_t, H, E, skip);
            else
                RL_LAUNCH(ctx, big_gates_tan_kernel, pw_grid, 256, 0, pl.tG, pl.R + t * HE, pl.U + t * HE, pl.N + t * HE, pl.HN + t * HE, hp_t,
                          pl.thp, pl.THNEW + t * HE, succ_t, H, E, skip);
        }
    }
    switch (mode) {
    case RL_PASS_STATS: RL_TRY(launch_head<RL_PASS_STATS>(ctx, a, pl, scal_part, head_blocks)); break;
    case RL_PASS_EVAL: RL_TRY(launch_head<RL_PASS_EVAL>(ctx, a, pl, scal_part, head_blocks)); break;
    case RL_PASS_GRAD: RL_TRY(launch_head<RL_PASS_GRAD>(ctx, a, pl, scal_part, head_blocks)); break;
    case RL_PASS_FVP: RL_TRY(launch_head<RL_PASS_FVP>(ctx, a, pl, scal_part, head_blocks)); break;
    case RL_PASS_VALUE: RL_TRY(launch_head<RL_PASS_VALUE>(ctx, a, pl, scal_part, head_blocks)); break;
    case RL_PASS_QLOSS: RL_TRY(launch_head<RL_PASS_QLOSS>(ctx, a, pl, scal_part, head_blocks)); break;
    case RL_PASS_PPO: RL_TRY(launch_head<RL_PASS_PPO>(ctx, a, pl, scal_part, head_blocks)); break;
    case RL_PASS_REINFORCE: RL_TRY(launch_head<RL_PASS_REINFORCE>(ctx, a, pl, scal_part, head_blocks)); break;
    default: return rl_fail(ctx, RL_ERR_INVALID_ARG, "rl_seq_big_pass_launch: bad mode %d", mode);
    }
    // ---- backward through time, then the weight gradients as two split-K GEMMs over all (t, e) ----
    if (backward) {
        const int o_lw = NG * H * F + NG * H * H + 2 * NG * H;
        RL_LAUNCH(ctx, big_zero_kernel, 256, 256, 0, pl.dh, HE, skip);
        if (lstm) RL_LAUNCH(ctx, big_zero_kernel, 256, 256, 0, pl.dc, HE, skip);
        for (int64_t t = (int64_t)T - 1; t >= 0; --t) {
            if (lstm)
                RL_LAUNCH(ctx, lstm_bwd_kernel, pw_grid, 256, 0, a.dzbuf + (uint64_t)t * A * E, a.theta, o_lw, a.act, pl.R + t * HE, pl.U + t * HE,
                          pl.N + t * HE, pl.HN + t * HE, pl.HNEW + t * HE, pl.CP + t * HE, a.succ + (uint64_t)t * E, pl.dh, pl.dc,
                          pl.D + (uint64_t)t * 4 * HE, pl.AV + t * HE, H, A, E, skip);
            else
                RL_LAUNCH(ctx, big_bwd_kernel, pw_grid, 256, 0, a.dzbuf + (uint64_t)t * A * E, a.theta, o_lw, a.act, pl.R + t * HE, pl.U + t * HE,
                          pl.N + t * HE, pl.HN + t * HE, pl.HNEW + t * HE, a.hbuf + t * HE, a.succ + (uint64_t)t * E, pl.dh,
                          pl.D + (uint64_t)t * 4 * HE, pl.AV + t * HE, H, A, E, skip);
            if (t > 0) {
                const float *D_t = pl.D + (uint64_t)t * 4 * HE;
                if (use_tc) {
                    bt::BtArgs g{};
                    g.src0 = D_t; g.src1 = D_t; g.src2 = D_t; g.k0 = 3 * H; g.k1 = 3 * H; g.K = 3 * H; g.nsteps = stB; g.wp = wpB; g.E = E;
                    g.out = pl.dh; g.skip_flag = skip;
                    RL_TRY((launch_tc<128, bt::EPI_ACC>(ctx, g)));
                } else {
                    RL_TRY(gemm_nn(ctx, WhT, NG * H, D_t, D_t, NG * H, E, pl.dh, E, nullptr, 1, H, E, NG * H, skip));
                }
            }
        }
        if (nt_tc) {
            float *ntpart = (float *)(base + o_ntpart);
            RL_CUDA(ctx, cudaMemsetAsync(ntpart, 0, nt_part_bytes, ctx->stream));
            static bool nt_configured = false;
            if (!nt_configured) {
                RL_CUDA(ctx, cudaFuncSetAttribute(bt::big_nt_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bt::nt_smem()));
                nt_configured = true;
            }
            bt::NtArgs na{};
            na.D = pl.D; na.src0 = a.obs; na.src1 = a.hbuf; na.rows0 = F; na.rows1 = H; na.T = T; na.E = E; na.part = ntpart;
            na.splits = nt_splits; na.nd = nt_nd; na.skip_flag = skip;
            RL_LAUNCH(ctx, bt::big_nt_tc_kernel, dim3((unsigned)nt_splits, 2), bt::BT_THREADS, bt::nt_smem(), na);
            RL_LAUNCH(ctx, bt::splitk_reduce_f32_kernel, (unsigned)rl_div_up(512 * bt::NT_ROWS_B, 256), 256, 0, ntpart, nt_splits * nt_nd, NB, dWc, skip);
        } else {
            dim3 gW((unsigned)rl_div_up(NB, NT_BN), (unsigned)rl_div_up(4 * H, NT_BM), (unsigned)splits);
            RL_LAUNCH(ctx, gemm_nt_splitk_kernel, gW, NT_THREADS, 0, pl.D, 4 * H, a.obs, F, a.hbuf, H, T, E, partW, NB, splits, skip);
            RL_LAUNCH(ctx, splitk_reduce_kernel, (unsigned)rl_div_up(4 * H * NB, 256), 256, 0, partW, splits, 4 * H * NB, dWc, skip);
        }
        dim3 gH((unsigned)rl_div_up(NH, NT_BN), (unsigned)rl_div_up(A, NT_BM), (unsigned)splits);
        RL_LAUNCH(ctx, gemm_nt_splitk_kernel, gH, NT_THREADS, 0, a.dzbuf, A, pl.AV, H, (const float *)nullptr, 0, T, E, partH, NH, splits, skip);
        RL_LAUNCH(ctx, splitk_reduce_kernel, (unsigned)rl_div_up(A * NH, 256), 256, 0, partH, splits, A * NH, dHead, skip);
    }
    if (lstm)
        RL_LAUNCH(ctx, lstm_assemble_kernel, 32, 256, 0, dWc, dHead, scal_part, head_blocks, F, H, A, backward ? 1 : 0, a.partials, skip);
    else
        RL_LAUNCH(ctx, big_assemble_kernel, 32, 256, 0, dWc, dHead, scal_part, head_blocks, F, H, A, backward ? 1 : 0, a.partials, skip);
    return RL_OK;
}

// SeqPacked::seq_packed over a stored trajectory (gru.rs:72-102 -> chain.rs:157-168) in the GEMM form: out f32 [T][A][E] (zeros
// on padding) and, when out_next is given, the module's output on the successor observation of every interrupted step
// (features.rs:139-185: one more step of the same sequence).  What rl_gae_seq needs from a hidden-128 critic.
rl_status rl_seq_big_forward(rl_ctx *ctx, int cell, const float *params, int F, int H, int A, int act, const float *obs,
                             const float *next_obs, const uint8_t *succ, uint64_t T, uint64_t E, float *out, float *out_next) {
    const int KP = F + H;
    const bool lstm = cell == RL_CELL_LSTM;
    const uint64_t HE = (uint64_t)H * E;
    auto al = [](size_t b) { return (b + 255) / 256 * 256; };
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += al(bytes); return o; };
    const size_t o_Wc = take((size_t)4 * H * KP * 4), o_bc = take((size_t)4 * H * 4), o_G = take(4 * HE * 4);
    const size_t o_tmp = take(4 * HE * 4), o_hn = take(HE * 4), o_h2 = take(HE * 4), o_ha = take(HE * 4), o_hb = take(HE * 4);
    const size_t o_ca = take(lstm ? HE * 4 : 0), o_cb = take(lstm ? HE * 4 : 0), o_c2 = take(lstm ? HE * 4 : 0);
    const bool use_tc = H == 128 && seq_tc_enabled() && !lstm;
    const int stW = (KP + 15) / 16;
    const size_t o_wpW = take(use_tc ? (size_t)stW * bt::bt_b_stage(512) : 0);
    char *base;
    RL_TRY(rl_ctx_scratch2(ctx, off + 256, (void **)&base));
    uint16_t *wpW = (uint16_t *)(base + o_wpW);
    float *Wc = (float *)(base + o_Wc), *bc = (float *)(base + o_bc), *G = (float *)(base + o_G), *tmp = (float *)(base + o_tmp);
    float *hnew = (float *)(base + o_hn), *h2 = (float *)(base + o_h2), *hcur = (float *)(base + o_ha), *hnxt = (float *)(base + o_hb);
    float *ccur = (float *)(base + o_ca), *cnxt = (float *)(base + o_cb), *c2 = (float *)(base + o_c2);
    const unsigned pw_grid = (unsigned)rl_div_up(HE, 256), e_grid = (unsigned)rl_div_up(E, 128);
    const int NG = rl_cell_gates(cell), o_lw = NG * H * F + NG * H * H + 2 * NG * H;
    const size_t hsmem = (size_t)(A * H + A) * sizeof(float);
    auto comb = lstm ? lstm_comb_kernel : big_comb_kernel;
    RL_LAUNCH(ctx, comb, 64, 256, 0, params, F, H, Wc, bc, (float *)nullptr);
    RL_LAUNCH(ctx, big_zero_kernel, 256, 256, 0, hcur, HE, (const int *)nullptr);
    if (lstm) RL_LAUNCH(ctx, big_zero_kernel, 256, 256, 0, ccur, HE, (const int *)nullptr);
    // one cell step over all lanes: gates into tmp, h' into hout (an LSTM's c' into cout), the next step's state (zero after an
    // episode's end) into hnext / cnext
    auto cell_fp32 = [&](const float *x, const float *hp, const float *cp, const uint8_t *succ_t, float *hout, float *cout, float *hnext,
                         float *cnext) -> rl_status {
        RL_TRY(gemm_nn(ctx, Wc, KP, x, hp, F, E, G, E, bc, 0, 4 * H, E, KP, nullptr));
        if (lstm)
            RL_LAUNCH(ctx, lstm_gates_kernel, pw_grid, 256, 0, G, cp, succ_t, tmp, tmp + HE, tmp + 2 * HE, tmp + 3 * HE, hout, cout, hnext,
                      cnext, H, E, (const int *)nullptr);
        else
            RL_LAUNCH(ctx, big_gates_kernel, pw_grid, 256, 0, G, hp, succ_t, tmp, tmp + HE, tmp + 2 * HE, tmp + 3 * HE, hout, hnext, H, E,
                      (const int *)nullptr);
        return RL_OK;
    };
    if (use_tc) RL_LAUNCH(ctx, bt::big_pieces_kernel, 128, 256, 0, Wc, KP, KP, (const float *)nullptr, 0, 0, 4 * H, stW, wpW);
    auto cell_tc = [&](const float *x, const float *hp, const uint8_t *succ_t, float *hout, float *hnext) -> rl_status {
        bt::BtArgs g{};
        g.src0 = x; g.src1 = hp; g.src2 = hp; g.k0 = F; g.k1 = KP; g.K = KP; g.nsteps = stW; g.wp = wpW; g.E = E; g.bias = bc;
        g.succ_t = succ_t; g.R = tmp; g.U = tmp + HE; g.Nn = tmp + 2 * HE; g.HN = tmp + 3 * HE; g.HNEW = hout; g.hnext = hnext;
        return launch_tc<512, bt::EPI_GATES>(ctx, g);
    };
    for (uint64_t t = 0; t < T; ++t) {
        const uint8_t *succ_t = succ + t * E;
        if (use_tc) {
            RL_TRY(cell_tc(obs + t * (uint64_t)F * E, hcur, succ_t, hnew, hnxt));
            RL_LAUNCH(ctx, big_head_out_kernel, e_grid, 128, hsmem, params, o_lw, act, hnew, succ_t, -1, out + t * (uint64_t)A * E, H, A, E);
            if (out_next) {
                RL_TRY(cell_tc(next_obs + t * (uint64_t)F * E, hnew, succ_t, h2, nullptr));
                RL_LAUNCH(ctx, big_head_out_kernel, e_grid, 128, hsmem, params, o_lw, act, h2, succ_t, (int)RL_INTERRUPT,
                          out_next + t * (uint64_t)A * E, H, A, E);
            }
            std::swap(hcur, hnxt);
            continue;
        }
        // the successor step of an interrupted episode continues from (h', c') before they are cut at the episode's end
        RL_TRY(cell_fp32(obs + t * (uint64_t)F * E, hcur, ccur, succ_t, hnew, lstm && out_next ? c2 : (float *)nullptr, hnxt, cnxt));
        RL_LAUNCH(ctx, big_head_out_kernel, e_grid, 128, hsmem, params, o_lw, act, hnew, succ_t, -1, out + t * (uint64_t)A * E, H, A, E);
        if (out_next) {
            RL_TRY(cell_fp32(next_obs + t * (uint64_t)F * E, hnew, c2, succ_t, h2, (float *)nullptr, (float *)nullptr, (float *)nullptr));
            RL_LAUNCH(ctx, big_head_out_kernel, e_grid, 128, hsmem, params, o_lw, act, h2, succ_t, (int)RL_INTERRUPT,
                      out_next + t * (uint64_t)A * E, H, A, E);
        }
        std::swap(hcur, hnxt);
        std::swap(ccur, cnxt);
    }
    return RL_OK;
}

// ---- one gru_cell over all lanes on the tensor cores, for the stepped rollout (gru.cu K8s): prepared = [Wc | bc | pieces] ----
bool rl_seq_big_cell_supports(int F, int H) { return H == 128 && F >= 1 && F <= 64 && seq_tc_enabled(); }

size_t rl_seq_big_prepared_bytes(int F, int H) {
    const int KP = F + H, stW = (KP + 15) / 16;
    auto al = [](size_t b) { return (b + 255) / 256 * 256; };
    return al((size_t)4 * H * KP * 4) + al((size_t)4 * H * 4) + al((size_t)stW * bt::bt_b_stage(512));
}

rl_status rl_seq_big_prepare(rl_ctx *ctx, const float *params, int F, int H, void *prepared) {
    const int KP = F + H, stW = (KP + 15) / 16;
    auto al = [](size_t b) { return (b + 255) / 256 * 256; };
    char *base = static_cast<char *>(prepared);
    float *Wc = (float *)base, *bc = (float *)(base + al((size_t)4 * H * KP * 4));
    uint16_t *wpW = (uint16_t *)(base + al((size_t)4 * H * KP * 4) + al((size_t)4 * H * 4));
    RL_LAUNCH(ctx, big_comb_kernel, 64, 256, 0, params, F, H, Wc, bc, (float *)nullptr);
    RL_LAUNCH(ctx, bt::big_pieces_kernel, 128, 256, 0, Wc, KP, KP, (const float *)nullptr, 0, 0, 4 * H, stW, wpW);
    return RL_OK;
}

rl_status rl_seq_big_cell(rl_ctx *ctx, const void *prepared, int F, int H, const float *x, const float *h, uint64_t E, float *hnew) {
    const int KP = F + H, stW = (KP + 15) / 16;
    auto al = [](size_t b) { return (b + 255) / 256 * 256; };
    const char *base = static_cast<const char *>(prepared);
    bt::BtArgs g{};
    g.src0 = x; g.src1 = h; g.src2 = h; g.k0 = F; g.k1 = KP; g.K = KP; g.nsteps = stW; g.E = E;
    g.bias = (const float *)(base + al((size_t)4 * H * KP * 4));
    g.wp = (const uint16_t *)(base + al((size_t)4 * H * KP * 4) + al((size_t)4 * H * 4));
    g.HNEW = hnew;
    return launch_tc<512, bt::EPI_CELL>(ctx, g);
}
