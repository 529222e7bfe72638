// ubench_step.cu -- latency floor of the CartPole step chain on one warp (round 2, VERDICT r1 item 1).
//   nvcc -gencode arch=compute_100a,code=sm_100a -O3 -std=c++17 -o build/ubench_step scripts/ubench_step.cu
// Prints clocks per dependent DADD / DMUL / DFMA / FFMA / SHFL / 64-bit select, and clocks per CartPoleEnv::step_fast call when
// one warp runs nothing else (the state chained through the step, the action taken from a state bit).
#include <cstdio>
#include <cstdint>
#include <cuda_runtime.h>

#include "../relearn_b200/csrc/envs.cuh"

template <int OP>
__global__ void lat_kernel(double a, double b, long long *out, double *sink, int iters) {
    double x = a + threadIdx.x * 1e-9;
    float xf = (float)x;
    const long long t0 = clock64();
#pragma unroll 1
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            if (OP == 0) x = __dadd_rn(x, b);
            if (OP == 1) x = __dmul_rn(x, b);
            if (OP == 2) x = fma(x, b, a);
            if (OP == 3) xf = fmaf(xf, (float)b, (float)a);
            if (OP == 4) x = __shfl_sync(0xffffffffu, x, (threadIdx.x + 1) & 31);
            if (OP == 5) x = (__double2hiint(x) & 1) ? __dadd_rn(x, b) : __dmul_rn(x, b);
            if (OP == 6) { double y; asm volatile("rcp.approx.ftz.f64 %0, %1;" : "=d"(y) : "d"(x)); x = y; }
            if (OP == 7) xf = (float)(double)xf + 1.0f, x = (double)xf;
        }
    }
    const long long t1 = clock64();
    if (threadIdx.x == 0) out[blockIdx.x] = t1 - t0;
    sink[blockIdx.x * blockDim.x + threadIdx.x] = x + xf;
}

// step_fast chained
__global__ void step_kernel(CartPoleEnv::Params p, long long *out, double *sink, int iters, int active_warp_stride) {
    using E = CartPoleEnv;
    E::State s;
    s.x = 0.01 + 1e-4 * threadIdx.x; s.xd = -0.02; s.th = 0.03; s.thd = 0.01;
    s.meta = 0x80000000u | 500u;
    const int warp = threadIdx.x >> 5;
    if (warp % active_warp_stride != 0) return;
    int term = 0;
    const long long t0 = clock64();
#pragma unroll 1
    for (int i = 0; i < iters; ++i) {
        const uint32_t action = (uint32_t)(__double2loint(s.x) >> 3) & 1u;
        const int sc = E::step_fast(p, s, action);
        if (sc != RL_CONTINUE) {
            term++;
            s.x = 0.01; s.xd = 0.0; s.th = 0.02; s.thd = 0.0; s.meta = 0x80000000u | 500u;
        }
    }
    const long long t1 = clock64();
    if ((threadIdx.x & 31) == 0) out[blockIdx.x * (blockDim.x / 32) + warp] = t1 - t0;
    sink[blockIdx.x * blockDim.x + threadIdx.x] = s.x + s.th + term;
}

// FFMA2: dependent latency (CHAINS = 1) and issue rate (CHAINS = 8 independent accumulators)
template <int CHAINS>
__global__ void ffma2_kernel(float a, float b, long long *out, double *sink, int iters) {
    float2 x[CHAINS];
#pragma unroll
    for (int c = 0; c < CHAINS; ++c) x[c] = make_float2(a + c + threadIdx.x * 1e-3f, a - c);
    const float2 m = make_float2(b, b * 0.999f), k = make_float2(a * 0.01f, a * 0.02f);
    const long long t0 = clock64();
#pragma unroll 1
    for (int i = 0; i < iters; ++i) {
#pragma unroll
        for (int j = 0; j < 16; ++j)
#pragma unroll
            for (int c = 0; c < CHAINS; ++c) x[c] = __ffma2_rn(x[c], m, k);
    }
    const long long t1 = clock64();
    if ((threadIdx.x & 31) == 0) out[threadIdx.x >> 5] = t1 - t0;
    float acc = 0.0f;
#pragma unroll
    for (int c = 0; c < CHAINS; ++c) acc += x[c].x + x[c].y;
    sink[blockIdx.x * blockDim.x + threadIdx.x] = acc;
}

// The policy chain of the warp-specialised rollout kernels (8 threads per env, weights in registers, 5 -> 128 -> logit
// difference) on its own: row from shared memory -> 40 + 8 FFMA2 -> butterfly over 8 lanes -> action to shared memory.
__global__ void policy_chain_kernel(long long *out, double *sink, int iters) {
    constexpr int PPL = 8;
    __shared__ float4 row[32][2];
    __shared__ uint32_t act[32];
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, grp = lane >> 3, sub = lane & 7, el = (4 * warp + grp) & 31;
    float4 wA[PPL], wB[PPL], wC[PPL];
    float2 wD[PPL];
    for (int u = 0; u < PPL; ++u) {
        const float f = 0.01f * (sub + 8 * u + 1);
        wA[u] = make_float4(f, -f, 0.5f * f, 0.3f - f); wB[u] = make_float4(-f, f, 0.25f * f, f - 0.1f);
        wC[u] = make_float4(f, 0.1f, 0.01f, -0.02f); wD[u] = make_float2(0.3f - f, f);
    }
    if (threadIdx.x < 32) { row[threadIdx.x][0] = make_float4(0.01f, 0.02f, -0.03f, 0.04f); row[threadIdx.x][1] = make_float4(1.0f, 0.0f, 0.0f, 0.0f); }
    __syncthreads();
    uint32_t action = 0, total = 0;
    const long long t0 = clock64();
#pragma unroll 1
    for (int i = 0; i < iters; ++i) {
        const volatile float *rp = reinterpret_cast<const volatile float *>(&row[el][0]);
        const float4 ov = make_float4(rp[0], rp[1], rp[2], rp[3]);
        const float4 tv = make_float4(rp[4], rp[5], rp[6], rp[7]);
        const float2 o0 = make_float2(ov.x + action, ov.x), o1 = make_float2(ov.y, ov.y), o2 = make_float2(ov.z, ov.z);
        const float2 o3 = make_float2(ov.w, ov.w), o4 = make_float2(tv.x, tv.x);
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
        for (int o = 4; o > 0; o >>= 1) d += __shfl_xor_sync(0xffffffffu, d, o);
        action = d < 0.013f ? 0u : 1u;
        if (sub == 0) *(volatile uint32_t *)&act[el] = action;
        __syncwarp();
        total += action;
    }
    const long long t1 = clock64();
    if (lane == 0) out[warp] = t1 - t0;
    sink[blockIdx.x * blockDim.x + threadIdx.x] = (double)total;
}

int main() {
    long long *out;
    double *sink;
    cudaMallocManaged(&out, 4096 * sizeof(long long));
    cudaMalloc(&sink, 1 << 20);
    const int iters = 2000;
    const char *names[] = {"DADD", "DMUL", "DFMA", "FFMA", "SHFL64", "DSEL(add|mul)", "RCP64H", "F2F roundtrip"};
#define LAT(OP)                                                        \
    lat_kernel<OP><<<1, 32>>>(1.000001, 0.9999999, out, sink, iters);  \
    cudaDeviceSynchronize();                                           \
    printf("%-16s %.2f clk per dependent op\n", names[OP], (double)out[0] / (iters * 16.0));
    LAT(0) LAT(1) LAT(2) LAT(3) LAT(4) LAT(5) LAT(6) LAT(7)
    CartPoleEnv::Params p{};
    p.gravity = 9.8; p.mass_cart = 1.0; p.mass_pole = 0.1; p.length_half_pole = 0.5; p.friction_cart = 0.01; p.friction_pole = 0.001;
    p.time_step = 0.02; p.action_force = 10.0; p.max_pos = 2.4; p.max_angle = 0.2094;
    p.total_weight = 1.1 * 9.8; p.inv_total_mass = 1.0 / 1.1; p.mass_length_pole = 0.05; p.reset_low = -0.05; p.reset_scale = 0.1;
    p.max_steps = 500; p.visible = 1;
    for (int warps = 1; warps <= 8; warps *= 2) {
        step_kernel<<<1, 32 * warps>>>(p, out, sink, 4000, 1);
        cudaDeviceSynchronize();
        printf("step, %d warps on one SM: %.1f clk per step (warp 0)\n", warps, (double)out[0] / 4000.0);
    }
    ffma2_kernel<1><<<1, 32>>>(1.0f, 0.5f, out, sink, iters);
    cudaDeviceSynchronize();
    printf("FFMA2 dependent: %.2f clk per op\n", (double)out[0] / (iters * 16.0));
    for (int warps = 1; warps <= 16; warps *= 2) {
        ffma2_kernel<8><<<1, 32 * warps>>>(1.0f, 0.5f, out, sink, iters);
        cudaDeviceSynchronize();
        printf("FFMA2 8 independent chains, %d warps on one SM: %.2f clk per FFMA2 (warp 0)\n", warps, (double)out[0] / (iters * 16.0 * 8.0));
    }
    for (int warps = 1; warps <= 16; warps *= 2) {
        policy_chain_kernel<<<1, 32 * warps>>>(out, sink, 2000);
        cudaDeviceSynchronize();
        printf("policy chain, %d warps on one SM: %.1f clk per iteration (warp 0)\n", warps, (double)out[0] / 2000.0);
    }
    policy_chain_kernel<<<1, 32 * 12>>>(out, sink, 2000);
    cudaDeviceSynchronize();
    printf("policy chain, 12 warps on one SM: %.1f clk per iteration (warp 0)\n", (double)out[0] / 2000.0);
    printf("%s\n", cudaGetErrorString(cudaGetLastError()));
    return 0;
}
