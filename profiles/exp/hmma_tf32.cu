// Throughput and latency of mma.sync.m16n8k8 TF32 (SASS HMMA.1688.F32.TF32) on the GPU it runs on.
//
//     nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -o hmma_tf32 hmma_tf32.cu && ./hmma_tf32
//
// Each warp runs `chains` independent accumulator chains of `iters` dependent MMAs (the accumulator is C and D of
// every MMA in its chain, as in mlp_logits of random_envs_b200/csrc/renv_mlp_policy.cuh, where a row tile has 8 such
// chains of 24).  One wave of CTAs of 128 threads, `ctas` per SM.  Prints one JSON line per configuration: HMMA per
// SM-clock (the SM clock measured with clock64 over the same window), the TF32 FLOP per SM-clock (2 * 16 * 8 * 8 =
// 2048 per HMMA) and, for one warp per SM with one chain, the dependent-issue latency in clocks.
// Driven by profiles/time_hmma_tf32.py, which also places the numbers beside the MLP rollout's.
#include <cstdio>
#include <cstdint>
#include <cuda_runtime.h>

__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1)
{
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

template <int kChains>
__global__ void __launch_bounds__(128) hmma_kernel(float *out, long long *cycles, int iters, float seed)
{
    uint32_t a[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) a[q] = __float_as_uint(seed * (1.0f + 0.001f * (threadIdx.x + q))) & 0xffffe000u;
    const uint32_t b0 = __float_as_uint(seed * 0.5f) & 0xffffe000u, b1 = __float_as_uint(seed * 0.25f) & 0xffffe000u;
    float acc[kChains][4];
#pragma unroll
    for (int c = 0; c < kChains; ++c)
#pragma unroll
        for (int q = 0; q < 4; ++q) acc[c][q] = 0.0f;
    __syncthreads();
    const long long t0 = clock64();
    for (int it = 0; it < iters; ++it) {
#pragma unroll
        for (int c = 0; c < kChains; ++c) mma_tf32(acc[c], a, b0, b1);
    }
    __syncthreads();
    const long long t1 = clock64();
    float s = 0.0f;
#pragma unroll
    for (int c = 0; c < kChains; ++c) s += acc[c][0] + acc[c][1] + acc[c][2] + acc[c][3];
    out[blockIdx.x * blockDim.x + threadIdx.x] = s;
    if (threadIdx.x == 0) cycles[blockIdx.x] = t1 - t0;
}

template <int kChains> void run(int sms, int ctas_per_sm, int threads, int iters, float *out, long long *cyc)
{
    const int grid = sms * ctas_per_sm;
    hmma_kernel<kChains><<<grid, threads>>>(out, cyc, iters / 8, 1.0f);      // warm-up
    cudaEvent_t e0, e1;
    cudaEventCreate(&e0); cudaEventCreate(&e1);
    cudaEventRecord(e0);
    hmma_kernel<kChains><<<grid, threads>>>(out, cyc, iters, 1.0f);
    cudaEventRecord(e1);
    cudaEventSynchronize(e1);
    float ms = 0.0f;
    cudaEventElapsedTime(&ms, e0, e1);
    static long long host[148 * 64];
    cudaMemcpy(host, cyc, sizeof(long long) * grid, cudaMemcpyDeviceToHost);
    double mean_cyc = 0.0;
    for (int i = 0; i < grid; ++i) mean_cyc += (double)host[i];
    mean_cyc /= grid;
    const double warps = (double)grid * threads / 32.0;
    const double hmma = warps * (double)iters * kChains;
    const double per_sm_clk = hmma / sms / mean_cyc;      // the timed window of each CTA: all CTAs of the wave overlap
    printf("{\"chains\": %d, \"warps_per_sm\": %d, \"iters\": %d, \"ms\": %.3f, \"sm_clock_mhz\": %.0f, "
           "\"hmma_per_sm_clk\": %.4f, \"tf32_flop_per_sm_clk\": %.1f, \"clk_per_dependent_hmma\": %.2f, \"err\": \"%s\"}\n",
           kChains, ctas_per_sm * threads / 32, iters, ms, mean_cyc / (ms * 1e3), per_sm_clk, per_sm_clk * 2048.0,
           mean_cyc / iters, cudaGetErrorString(cudaGetLastError()));
    cudaEventDestroy(e0); cudaEventDestroy(e1);
}

int main()
{
    int dev = 0, sms = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    float *out; long long *cyc;
    cudaMalloc(&out, sizeof(float) * sms * 16 * 128);
    cudaMalloc(&cyc, sizeof(long long) * sms * 16);
    const int iters = 1 << 15;
    run<1>(sms, 1, 32, iters, out, cyc);                   // one warp per SM, one chain: dependent latency
    for (int c : {1, 2, 3, 4, 8, 16}) {
        run<1>(sms, c, 128, iters, out, cyc);
        run<2>(sms, c, 128, iters, out, cyc);
        run<4>(sms, c, 128, iters, out, cyc);
        run<8>(sms, c, 128, iters, out, cyc);
    }
    cudaFree(out); cudaFree(cyc);
    return 0;
}
