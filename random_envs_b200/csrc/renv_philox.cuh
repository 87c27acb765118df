// Counter-based RNG for the DR hot path: Philox4x32-10 (Salmon et al., SC'11) plus the
// framework's draw contract (DESIGN.md "RNG contract").
//
// The reference draws xi from the process-global numpy/scipy state (random_env.py:151,161,180)
// and s0 from a per-env RandomState (random_cartpole.py:227) -- a serial, stateful design.  Here
// every random number is a pure function of
//     key     = (seed lo, seed hi)
//     counter = (id[31:0], id[47:32] | tick[47:32] << 16, tick[31:0], purpose << 24 | slot)
// where `id` is the GLOBAL env (or sample) index and `tick` identifies the episode: it is the value of
// the env's step clock at the launch that (re)started the episode -- a host-side counter that advances
// by one per step / reset call and by K per K-step rollout.  An env starts at most one episode per tick,
// so (seed, id, tick) is unique per episode, needs NO per-env RNG state in HBM (a per-env episode
// counter would have to be loaded before the first Philox round: a dependent DRAM round trip inside the
// reset path), and is independent of launch geometry and of how envs are sharded across GPUs.
#pragma once
#include <stdint.h>

namespace renv {

enum Purpose : uint32_t { kInit = 0, kXi = 1, kAction = 2, kTasks = 3, kObs = 4, kPolicySample = 5 };

__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k)
{
    constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(M0, c.x), lo0 = M0 * c.x;
        const uint32_t hi1 = __umulhi(M1, c.z), lo1 = M1 * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        k.x += W0;
        k.y += W1;
    }
    return c;
}

// The same function with the ten round keys precomputed (a loop over many counters with one key: the samplers).
struct PhiloxKeys { uint32_t x[10], y[10]; };
__host__ __device__ __forceinline__ PhiloxKeys philox_keys(uint32_t kx, uint32_t ky)
{
    constexpr uint32_t W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
    PhiloxKeys ks;
#pragma unroll
    for (int r = 0; r < 10; ++r) { ks.x[r] = kx + (uint32_t)r * W0; ks.y[r] = ky + (uint32_t)r * W1; }
    return ks;
}
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, const PhiloxKeys &ks)
{
    constexpr uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u;
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(M0, c.x), lo0 = M0 * c.x;
        const uint32_t hi1 = __umulhi(M1, c.z), lo1 = M1 * c.z;
        c = make_uint4(hi1 ^ c.y ^ ks.x[r], lo1, hi0 ^ c.w ^ ks.y[r], lo0);
    }
    return c;
}

// One 128-bit block of the stream (seed, id, tick, purpose); slot = attempt * 16 + dim_block.
__device__ __forceinline__ uint4 draw_block(uint64_t seed, uint64_t id, uint64_t tick, uint32_t purpose, uint32_t slot)
{
    const uint32_t c1 = ((uint32_t)(id >> 32) & 0xffffu) | (((uint32_t)(tick >> 32) & 0xffffu) << 16);
    return philox4x32_10(make_uint4((uint32_t)id, c1, (uint32_t)tick, (purpose << 24) | slot),
                         make_uint2((uint32_t)seed, (uint32_t)(seed >> 32)));
}

// U[0,1) with 24 (float) / 53 (double, numpy's recipe) random bits.
__device__ __forceinline__ float u01(uint32_t r) { return (float)(r >> 8) * (1.0f / 16777216.0f); }
__device__ __forceinline__ double u01(uint32_t hi, uint32_t lo)
{
    return __dmul_rn(__dadd_rn(__dmul_rn((double)(hi >> 5), 67108864.0), (double)(lo >> 6)),
                     1.0 / 9007199254740992.0);
}
// (0,1] variants for log() in Box-Muller.
__device__ __forceinline__ float u01_open0(uint32_t r) { return (float)((r >> 8) + 1u) * (1.0f / 16777216.0f); }
__device__ __forceinline__ double u01_open0(uint32_t hi, uint32_t lo)
{
    return __dmul_rn(__dadd_rn(__dadd_rn(__dmul_rn((double)(hi >> 5), 67108864.0), (double)(lo >> 6)), 1.0),
                     1.0 / 9007199254740992.0);
}

// Per-type packing of one Philox block: 4 floats or 2 doubles.
template <typename T> struct Pack;
template <> struct Pack<float> {
    static constexpr int kPerBlock = 4;
    __device__ static __forceinline__ void uniforms(uint4 r, float u[4])
    {
        u[0] = u01(r.x); u[1] = u01(r.y); u[2] = u01(r.z); u[3] = u01(r.w);
    }
    // off + (hi - lo) * u with u = (r >> 8) * 2^-24.  `scale` arrives PRE-MULTIPLIED by 2^-24 (uniform_scale):
    // a power-of-two factor is exact, so fma(scale, (float)(r >> 8), off) has the same real argument -- hence the
    // same rounded result -- as fma(hi - lo, u, off), in one instruction less per value.
    static constexpr float kUniformScale = 1.0f / 16777216.0f;
    __device__ static __forceinline__ float uniform_scale(float width) { return width * kUniformScale; }
    __device__ static __forceinline__ void uniform_affine(uint4 r, const float scale[4], const float off[4], float out[4])
    {
        out[0] = fmaf(scale[0], (float)(r.x >> 8), off[0]);
        out[1] = fmaf(scale[1], (float)(r.y >> 8), off[1]);
        out[2] = fmaf(scale[2], (float)(r.z >> 8), off[2]);
        out[3] = fmaf(scale[3], (float)(r.w >> 8), off[3]);
    }
    // 4 standard normals: Box-Muller on the pairs (x,y) and (z,w), both branches used
    __device__ static __forceinline__ void normals(uint4 r, float z[4])
    {
        float s, c;
        float rad = sqrtf(-2.0f * logf(u01_open0(r.x)));
        sincospif(2.0f * u01(r.y), &s, &c);
        z[0] = rad * c; z[1] = rad * s;
        rad = sqrtf(-2.0f * logf(u01_open0(r.z)));
        sincospif(2.0f * u01(r.w), &s, &c);
        z[2] = rad * c; z[3] = rad * s;
    }
};
template <> struct Pack<double> {
    static constexpr int kPerBlock = 2;
    __device__ static __forceinline__ void uniforms(uint4 r, double u[2])
    {
        u[0] = u01(r.x, r.y); u[1] = u01(r.z, r.w);
    }
    // numpy: low + (high - low) * u, separately rounded
    __device__ static __forceinline__ double uniform_scale(double width) { return width; }
    __device__ static __forceinline__ void uniform_affine(uint4 r, const double scale[2], const double off[2], double out[2])
    {
        double u[2];
        uniforms(r, u);
        out[0] = __dadd_rn(off[0], __dmul_rn(scale[0], u[0]));
        out[1] = __dadd_rn(off[1], __dmul_rn(scale[1], u[1]));
    }
    __device__ static __forceinline__ void normals(uint4 r, double z[2])
    {
        double s, c;
        const double rad = sqrt(-2.0 * log(u01_open0(r.x, r.y)));
        sincospi(2.0 * u01(r.z, r.w), &s, &c);
        z[0] = rad * c; z[1] = rad * s;
    }
};

}  // namespace renv
