// sample_tasks(n) for dr_type 'fullgaussian' (random_env.py:192-198 + denormalize_parameters :205-220), dim 17..32,
// fp32, with the contraction on the 5th-generation tensor cores:
//
//     X (128 samples x 32) = Z (128 x 32 standard normals) . F^T (32 x 32),   F F^T = cov
//
// is the one GEMM-shaped piece of the hot path (2 dim^2 FLOPs per sample: on CUDA cores it made the 30-dim sampler
// FMA-bound at 0.20 of the HBM rate, round-1 verdict).  Per 128-sample tile of a persistent CTA (128 threads, one per
// sample; a 256-thread variant in which threads t and t + 128 share TMEM lane t and split the k / d range in halves
// was measured slower: 1.17 vs 1.03 ms for 2^24 x 30 -- the work per sample is the same and the barriers double):
//
//   1. the thread of sample t draws its 32 normals (the SAME Philox blocks and Box-Muller as the CUDA-core
//      kernel: draw_block(seed, id, call, kTasks, j), j = 0..7) and write them -- split into a TF32 head and a TF32
//      tail, z = z_hi + z_lo -- straight from registers into TENSOR MEMORY with tcgen05.st: row t of the A operand
//      is TMEM lane t, element k is column k.  Z never touches shared or global memory.
//   2. one thread issues 12 tcgen05.mma.kind::tf32 (M = 128, N = 32, K = 8; A from TMEM, B = F from shared memory
//      through a K-major no-swizzle matrix descriptor): for each of the 4 K-steps  D += Z_lo F_hi,  D += Z_hi F_lo,
//      D += Z_hi F_hi  ("3xTF32": the dropped Z_lo F_lo term is 2^-22 relative, i.e. fp32-grade products with fp32
//      accumulation in TMEM), then tcgen05.commit -> mbarrier.
//   3. the threads read their sample's results back with tcgen05.ld (lane t = sample t), add the
//      mean, clip to [0, 4], denormalise to the search bounds, and each lane quadrant writes its 32 rows as one
//      contiguous span.  The accumulator is double-buffered: the epilogue of tile i-1 runs while the tensor core
//      works on tile i, and the wait for tile i's MMAs sits after the NEXT tile's normals have been drawn.
//
// TMEM per CTA: 32 (Z_hi) + 32 (Z_lo) + 2 x 32 (D) = 128 columns: 4 CTAs per SM share the 512 columns.  (One
// accumulator, 64 + 32 columns and 5 CTAs per SM, measured 0.928 vs 0.939 ms for 2^24 x 30, +1 %: occupancy is not what
// holds the kernel back.)
// Tolerance against the fp32 FMA-chain kernel (same draws): <= 4e-6 of the search-bound width (tests/test_gpu_fullgaussian.py).
#pragma once
#include "renv_kernels.cuh"

namespace renv {

constexpr int kFgTile = 128;            // samples per tile = MMA M = TMEM lanes
constexpr int kFgThreads = 128;         // one thread per sample
constexpr int kFgCtas = 4;              // resident CTAs per SM: 4 x 128 TMEM columns
constexpr int kFgTmemCols = 128;        // Z_hi 32 + Z_lo 32 + two accumulators of 32
constexpr uint32_t kFgColZhi = 0, kFgColZlo = 32, kFgColD = 64;

struct __align__(128) FgTcSmem {
    float b_hi[32 * 32];                // F as the B operand, K-major core-matrix layout (see fg_b_index)
    float b_lo[32 * 32];
    float stage[kFgTile * 32];          // per lane quadrant: 32 rows of `dim` values, contiguous
    unsigned long long mbar;
    uint32_t tmem_base;
    uint32_t failed;
};

// K-major, no swizzle ("interleave") canonical layout of a 32 (N) x 32 (K) fp32 operand: 8-row x 16-byte core matrices,
// rows 16 bytes apart; the next core matrix along K is LBO = 128 bytes on, the next 8 rows SBO = 1024 bytes on.
__host__ __device__ constexpr int fg_b_index(int n, int k) { return (n >> 3) * 256 + (k >> 2) * 32 + (n & 7) * 4 + (k & 3); }

// tcgen05 shared-memory matrix descriptor: start address, leading / stride byte offsets (all >> 4), version 1 (sm_100),
// no swizzle, base offset 0.
__device__ __forceinline__ uint64_t fg_smem_desc(const void *p)
{
    const uint32_t a = (uint32_t)__cvta_generic_to_shared(p);
    return (uint64_t)((a >> 4) & 0x3fffu) | ((uint64_t)(128u >> 4) << 16) | ((uint64_t)(1024u >> 4) << 32) | (1ull << 46);
}
// Instruction descriptor of kind::tf32: D = F32 (bits 4-5 = 1), A = B = TF32 (bits 7-9, 10-12 = 2), both K-major,
// N >> 3 at bits 17-22, M >> 4 at bits 24-28.
constexpr uint32_t kFgIdesc = (1u << 4) | (2u << 7) | (2u << 10) | ((32u >> 3) << 17) | ((128u >> 4) << 24);

__device__ __forceinline__ void fg_mma(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, bool accumulate)
{
    const uint32_t acc = accumulate ? 1u : 0u, zero = 0u;
    asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
                 "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, {%5, %5, %5, %5}, p;\n\t}\n"
                 :: "r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(kFgIdesc), "r"(acc), "r"(zero) : "memory");
}
__device__ __forceinline__ void fg_tmem_st8(uint32_t taddr, const float *v)
{
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 :: "r"(taddr), "r"(__float_as_uint(v[0])), "r"(__float_as_uint(v[1])), "r"(__float_as_uint(v[2])),
                    "r"(__float_as_uint(v[3])), "r"(__float_as_uint(v[4])), "r"(__float_as_uint(v[5])),
                    "r"(__float_as_uint(v[6])), "r"(__float_as_uint(v[7])) : "memory");
}
__device__ __forceinline__ void fg_tmem_ld32(uint32_t taddr, float *v)
{
    uint32_t r[32];
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x32.b32 "
                 "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
                 "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                   "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
                   "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
                   "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
                 : "r"(taddr) : "memory");
    asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
    for (int k = 0; k < 32; ++k) v[k] = __uint_as_float(r[k]);
}
__global__ void __launch_bounds__(kFgThreads, kFgCtas)
dr_sample_fullgaussian_tc_kernel(float *__restrict__ out, int64_t n, const __grid_constant__ FullGaussCfg<float> cfg,
                                 const __grid_constant__ PhiloxKeys ks, uint64_t sample_id0, uint32_t call,
                                 unsigned long long *counters)
{
    __shared__ FgTcSmem sm;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int dim = cfg.dim;

    // ---- set-up: F -> B operand (TF32 head / tail), mbarrier, TMEM allocation ------------------------------------
    for (int e = tid; e < 32 * 32; e += kFgThreads) {
        const int d = e >> 5, k = e & 31;                       // B[n = d][k] = F[d][k] = ft[k][d] (zero beyond dim)
        const float f = cfg.ft[k * 32 + d];
        const float hi = __uint_as_float(__float_as_uint(f) & 0xffffe000u);
        sm.b_hi[fg_b_index(d, k)] = hi;
        sm.b_lo[fg_b_index(d, k)] = f - hi;                     // exact; the tensor core keeps its leading 11 bits
    }
    if (tid == 0) {
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" :: "r"((uint32_t)__cvta_generic_to_shared(&sm.mbar)));
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        sm.failed = 0;
    }
    if (warp == 0) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     :: "r"((uint32_t)__cvta_generic_to_shared(&sm.tmem_base)), "n"(kFgTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");           // B was written through the generic proxy
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t tmem = sm.tmem_base;
    const uint32_t tmem_d = tmem + kFgColD;                                // two accumulators behind Z
    const int quad = warp;                                                 // TMEM lane quadrant
    const uint32_t lane_base = tmem + ((uint32_t)(quad * 32) << 16);       // this warp's 32 TMEM lanes
    const uint32_t lane_base_d = tmem_d + ((uint32_t)(quad * 32) << 16);
    const uint64_t desc_hi = fg_smem_desc(sm.b_hi), desc_lo = fg_smem_desc(sm.b_lo);
    const uint32_t mbar = (uint32_t)__cvta_generic_to_shared(&sm.mbar);

    auto wait_mma = [&](uint32_t parity) {      // bounded (an encoding error must not hang the GPU): ~0.2 s, then give up loudly
        uint32_t ready = 0;
        for (int spin = 0; !ready && spin < (1 << 22); ++spin)
            asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                         : "=r"(ready) : "r"(mbar), "r"(parity) : "memory");
        if (!ready) sm.failed = 1;
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    };
    // rows of tile `tile` out of accumulator `buf`: clip, denormalise, and write the quadrant's 32 rows as one span
    auto epilogue = [&](int64_t tile, int buf) {
        float x[32];
        fg_tmem_ld32(lane_base_d + 32 * buf, x);
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        float *rows = sm.stage + quad * 32 * 32;
        float *row = rows + lane * dim;
#pragma unroll
        for (int d = 0; d < 32; ++d) {
            // (clip(mean + x, 0, 4) * width) / 4 + lo (random_env.py:194-198, 205-220) in two instructions: scaling by
            // 1/4 is exact and commutes with rounding, so sat(x / 4 + mean / 4) == clip(fl(mean + x), 0, 4) / 4 and
            // fl(q * width) == fl(p * width) / 4 bit for bit; the host passes mean / 4 and width = hi - lo
            const float q4 = __saturatef(fmaf(x[d], 0.25f, cfg.mean[d]));
            if (d < dim) row[d] = fmaf(q4, cfg.hi[d], cfg.lo[d]);
        }
        __syncwarp();
        const int64_t quad_first = tile * kFgTile + quad * 32;
        const int nrows = (int)max((int64_t)0, min((int64_t)32, n - quad_first));
        const int total = nrows * dim;
        float *dst = out + quad_first * dim;                        // 32 * dim * 4 bytes is a multiple of 128
        const int nvec = total / 4;
        for (int q = lane; q < nvec; q += 32)
            reinterpret_cast<uint4 *>(dst)[q] = reinterpret_cast<const uint4 *>(rows)[q];
        for (int q = nvec * 4 + lane; q < total; q += 32) dst[q] = rows[q];
        __syncwarp();                                               // the stage may be rewritten
    };

    const int64_t num_tiles = (n + kFgTile - 1) / kFgTile;
    int it = 0;
    int64_t prev_tile = -1;
    for (int64_t tile = blockIdx.x; tile < num_tiles; tile += gridDim.x, ++it) {
        const int64_t i = tile * kFgTile + quad * 32 + lane;
        const uint64_t id = sample_id0 + (uint64_t)i;

        // ---- 1. this thread's normals (Philox blocks 0 .. 7), split into TF32 head and tail
        float hi[32], lo[32];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            float z[4];
            // draw_block(seed, id, call, kTasks, j) with the round keys as constant-bank operands
            const uint32_t c1 = (uint32_t)(id >> 32) & 0xffffu, c3 = ((uint32_t)kTasks << 24) | (uint32_t)j;
            Num<float>::normals(philox4x32_10(make_uint4((uint32_t)id, c1, call, c3), ks), z);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                hi[4 * j + q] = __uint_as_float(__float_as_uint(z[q]) & 0xffffe000u);
                lo[4 * j + q] = z[q] - hi[4 * j + q];
            }
        }
        // the previous tile's MMAs must have read Z before it is overwritten (they finished long ago: they ran while
        // the normals above were drawn); its accumulator is then ready for the epilogue further down
        if (it > 0) wait_mma((uint32_t)(it - 1) & 1u);
#pragma unroll
        for (int q = 0; q < 32; q += 8) {
            fg_tmem_st8(lane_base + kFgColZhi + q, hi + q);
            fg_tmem_st8(lane_base + kFgColZlo + q, lo + q);
        }
        asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
        asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
        __syncthreads();

        // ---- 2. D[it & 1] = Z F^T on the tensor core
        if (tid == 0) {
            asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
            const uint32_t d_col = tmem_d + 32 * (it & 1);
#pragma unroll
            for (int s = 0; s < 4; ++s) {               // K-step s: columns 8 s .. 8 s + 7 of Z, 256 bytes further into B
                const uint64_t off = (uint64_t)((256u * s) >> 4);
                fg_mma(d_col, tmem + kFgColZlo + 8 * s, desc_hi + off, s > 0);
                fg_mma(d_col, tmem + kFgColZhi + 8 * s, desc_lo + off, true);
                fg_mma(d_col, tmem + kFgColZhi + 8 * s, desc_hi + off, true);
            }
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" :: "r"(mbar) : "memory");
        }

        // ---- 3. epilogue of the PREVIOUS tile while the tensor core works on this one
        if (it > 0) epilogue(prev_tile, (it - 1) & 1);
        prev_tile = tile;
    }
    if (it > 0) {
        wait_mma((uint32_t)(it - 1) & 1u);
        epilogue(prev_tile, (it - 1) & 1);
    }

    // ---- teardown
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (tid == 0 && sm.failed && counters) atomicAdd(counters + kCounterOrderTimeout, 1ull);
    if (warp == 0)
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem), "n"(kFgTmemCols) : "memory");
}

}  // namespace renv
