// sm_100a kernels of the DR cart-pole hot path.  Launched only through the C ABI in renv_abi.cu.
//
// Memory design (HBM3e-bound single step): structure-of-arrays state (4, ld), one row per env for xi
// (n, 4); one thread owns V consecutive envs (V = 4 floats / 2 doubles = one 128-bit access per state
// row and per xi row), so every global access of the main path is a 128-bit LDG.E.128 / STG.E.128: per env-step 37 B read + 25 B written in fp32 (62 B),
// 69 + 45 = 114 B in fp64 (DESIGN.md "algorithmic bytes").  All loads are issued before the first
// use (10 independent 128-bit requests per thread in flight).  Auto-reset and the DR resample are
// fused into the same kernel: only envs that finished rewrite `xi`, and nothing is loaded for a reset
// (Philox is keyed by the launch's clock tick, not by a per-env counter in HBM).
#pragma once
#include <cuda_runtime.h>
#include "renv_cartpole.cuh"

namespace renv {

template <typename T> struct VecTraits;
template <> struct VecTraits<float> {
    static constexpr int V = 4;
    using Real = float4; using Int = int4; using Byte = uchar4; using Half = ushort4;
};
template <> struct VecTraits<double> {
    static constexpr int V = 2;
    using Real = double2; using Int = int2; using Byte = uchar2; using Half = ushort2;
};

__device__ __forceinline__ bool full_tile(int64_t block0, int64_t n, int tile) { return block0 + tile <= n; }

template <typename Vec, typename S, int V> __device__ __forceinline__ void vload(S (&dst)[V], const S *src)
{
    static_assert(sizeof(Vec) == sizeof(S) * V, "vector width");
    const Vec v = *reinterpret_cast<const Vec *>(src);
    const S *e = reinterpret_cast<const S *>(&v);
#pragma unroll
    for (int k = 0; k < V; ++k) dst[k] = e[k];
}
template <typename Vec, typename S, int V> __device__ __forceinline__ void vstore(S *dst, const S (&src)[V])
{
    Vec v;
    S *e = reinterpret_cast<S *>(&v);
#pragma unroll
    for (int k = 0; k < V; ++k) e[k] = src[k];
    *reinterpret_cast<Vec *>(dst) = v;
}

// xi is array-of-rows, (n, 4) row-major: one 16-byte (float) / 32-byte (double) row per env, so that a reset
// dirties ONE 32-byte DRAM sector instead of one in each of four SoA rows (ncu, 2^24 envs: +80 MB of write-backs
// per step with SoA xi).  Reads stay sector-exact: a thread's V rows are contiguous and the warp's span is one block.
__device__ __forceinline__ Xi<float> load_xi(const float *xi, int64_t i)
{
    const float4 v = *reinterpret_cast<const float4 *>(xi + 4 * i);
    return Xi<float>{ v.x, v.y, v.z, v.w };
}
__device__ __forceinline__ Xi<double> load_xi(const double *xi, int64_t i)
{
    const double2 a = *reinterpret_cast<const double2 *>(xi + 4 * i), b = *reinterpret_cast<const double2 *>(xi + 4 * i + 2);
    return Xi<double>{ a.x, a.y, b.x, b.y };
}
__device__ __forceinline__ void store_xi(float *xi, int64_t i, const Xi<float> &p)
{
    *reinterpret_cast<float4 *>(xi + 4 * i) = make_float4(p.gravity, p.cart_mass, p.pole_mass, p.pole_length);
}
__device__ __forceinline__ void store_xi(double *xi, int64_t i, const Xi<double> &p)
{
    *reinterpret_cast<double2 *>(xi + 4 * i) = make_double2(p.gravity, p.cart_mass);
    *reinterpret_cast<double2 *>(xi + 4 * i + 2) = make_double2(p.pole_mass, p.pole_length);
}

template <typename T> struct EnvPtrs {
    T *state; T *xi; int32_t *elapsed; uint32_t *episode; int32_t *beyond;
    uint16_t *elapsed16;      // lean step only: the TimeLimit counter as uint16 (then `elapsed` may be nullptr)
    uint32_t *progress;       // tile-granular step ordering (see cartpole_step_kernel); nullptr: the stream orders steps
    int64_t n, ld; uint64_t env_id0, seed;
    T *obs; T noise_std;      // "Noisy" variants: obs (4, ld) = state + noise_std * N(0, I); obs == nullptr: obs IS state
};

// RandomCartPoleEnv.reset (+ set_random_task) of env i at clock `tick`; scalar stores.
template <typename T>
__device__ __forceinline__ unsigned reset_env(const EnvPtrs<T> &env, const DrCfg4<T> &dr, int64_t i, uint64_t tick, uint64_t seed)
{
    const int64_t ld = env.ld;
    const uint64_t id = env.env_id0 + (uint64_t)i;
    State<T> st;
    init_state(st, seed, id, tick);
    env.state[0 * ld + i] = st.x; env.state[1 * ld + i] = st.x_dot;
    env.state[2 * ld + i] = st.theta; env.state[3 * ld + i] = st.theta_dot;
    if (env.obs) {                                         // noisy observation of the reset state (_get_obs in reset_model)
        T o[4];
        add_obs_noise(st, env.noise_std, seed, id, tick, 1u, o);
        env.obs[0 * ld + i] = o[0]; env.obs[1 * ld + i] = o[1]; env.obs[2 * ld + i] = o[2]; env.obs[3 * ld + i] = o[3];
    }
    unsigned viol = 0;
    if (dr.dr_type != kDrNone) {
        Xi<T> xi = { T(0), T(0), T(0), T(0) };
        viol = sample_xi(xi, dr, seed, id, tick);
        store_xi(env.xi, i, xi);
    }
    if (env.episode) atomicAdd(env.episode + i, 1u);      // optional episode count: fire-and-forget RED, no load stall
    return viol;
}

// Episode log (include/renv.h renv_episode_log): a per-env ring of `capacity` records.  Record r of env i lives at
// row (r mod capacity) * ld + i of every field; count[i] is the number of records env i has written.  Only the
// thread that resets env i writes them, so no atomics are needed and the content is independent of launch geometry.
template <typename T> struct LogPtrs {
    T *xi; T *final_state; int32_t *length; uint8_t *truncated; int64_t *end_tick; int32_t *count;
    uint32_t capacity;
};

// the termination test of dynamics() (:200-205), for a record whose episode ended: truncated = !this && length >= limit
template <typename T> __device__ __forceinline__ bool beyond_thresholds(const State<T> &s)
{
    return s.x < -(T)kXThreshold || s.x > (T)kXThreshold || s.theta < -(T)kThetaThreshold || s.theta > (T)kThetaThreshold;
}

// Writes record number `count` of env i (the caller stores count + 1).
template <typename T>
__device__ __forceinline__ void log_episode(const LogPtrs<T> &log, int64_t ld, int64_t i, uint32_t count, const Xi<T> &xi,
                                            const State<T> &s, int32_t length, bool truncated, uint64_t tick)
{
    const int64_t r = (int64_t)(count % log.capacity) * ld + i;
    store_xi(log.xi, r, xi);
    store_xi(log.final_state, r, Xi<T>{ s.x, s.x_dot, s.theta, s.theta_dot });      // the same 4-wide row layout
    log.length[r] = length;
    log.truncated[r] = truncated ? 1 : 0;
    log.end_tick[r] = (int64_t)tick;
}

// ------------------------------------------------------------------------------------------------
// Single step: RandomCartPoleEnv.step + TimeLimit.step + SyncVectorEnv auto-reset (+ set_random_task)
// ------------------------------------------------------------------------------------------------
// Device counters the host checks at its next synchronisation point (include/renv.h RENV_NUM_COUNTERS).
enum Counter : int { kCounterGaussian = 0, kCounterBadAction = 1, kCounterOrderTimeout = 2 };

__device__ __forceinline__ uint32_t ld_acquire_gpu(const uint32_t *p)
{
    uint32_t v;
    asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_release_gpu(uint32_t *p, uint32_t v)
{
    asm volatile("st.release.gpu.global.u32 [%0], %1;" :: "l"(p), "r"(v) : "memory");
}
// L2 prefetch of a contiguous span (1-D bulk form: one instruction, no register or shared-memory destination).
__device__ __forceinline__ void prefetch_l2(const void *p, uint32_t bytes)
{
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" :: "l"(p), "r"(bytes) : "memory");
}
constexpr int kOrderSpins = 1 << 21;       // x ~40 ns: ~0.1 s, then the CTA proceeds and raises kCounterOrderTimeout

template <typename T> struct StepArgs {
    EnvPtrs<T> env;
    const uint8_t *action; T *reward; uint8_t *done; uint8_t *truncated;
    int euler, max_steps;
    uint64_t tick;
    DrCfg4<T> dr;
    unsigned long long *counters;   // [kCounterGaussian], [kCounterBadAction]; may be nullptr
};

constexpr int kStepThreads = 256;          // x V envs = RENV_TILE_ENVS_F32 / _F64 (include/renv.h; checked in renv_abi.cu)
template <typename T> constexpr int kStepMinCtas = sizeof(T) == 4 ? 4 : 3;     // resident CTAs per SM (register cap)

// Tiles a CTA may own in one launch (tickets are kept in shared memory); the launcher sizes the grid accordingly.
// kAutoReset = true is the hot kernel.  Finished envs are NOT reset by the thread that owns them (that would
// run the ~250-instruction Philox/sampling path once per warp per finished lane with ~1 active lane): their
// CTA-local indices are appended to a shared-memory list and, after one __syncthreads, the first `count`
// threads of the CTA each reset one env at full lane utilisation, overwriting the owner's stores.
//
// kLean (auto-reset only): the TimeLimit counter is a.env.elapsed16 (uint16: 2 + 2 B instead of 4 + 4 B per env-step); the
// reward -- identically 1.0 under auto-reset, random_cartpole.py:207-212 -- is not written when a.reward == nullptr
// (any variant).  Together: 54 instead of 62 B per fp32 env-step.  State / done / truncated are bit-identical.
//
// Ordering between consecutive steps of one stream (a tile = one CTA = kStepThreads * V consecutive envs):
//
// (a) env.progress == nullptr: GRID-granular.  Programmatic dependent launch (the launcher sets
//     cudaLaunchAttributeProgrammaticStreamSerialization): griddepcontrol.wait -- before the first global access -- until
//     the PREVIOUS grid of the stream has completed and flushed; further down this grid lets the NEXT one be scheduled
//     into SM slots as it drains.  No-ops without the attribute.
// (b) env.progress != nullptr: TILE-granular.  A step of env i depends on the previous step of env i and on nothing
//     else, so the grid-wide wait is replaced by two words per tile:
//         progress[2 b]      tickets handed out for tile b   (atomicAdd at CTA entry)
//         progress[2 b + 1]  steps completed on tile b       (st.release after the CTA's last store)
//     CTA b takes ticket t and steps its tile as soon as progress[2 b + 1] == t.  The ticket is taken BEFORE the CTA
//     executes griddepcontrol.launch_dependents and the next grid of the stream cannot start before every CTA of this
//     one has done so, hence tickets follow launch order; and every predecessor CTA is resident or finished when a
//     CTA spins, hence no deadlock.  Kernels of the same stream then overlap: the ~2.3 us launch-to-launch bubble of
//     (a) (drain + flush + first DRAM round trip) shrinks to the CTA's own ticket round trip, during which the tile is
//     pulled from HBM into L2 by bulk prefetches (UBLKPF: no registers, no shared memory), and steps of DIFFERENT env
//     batches issued round-robin on one stream do not wait for each other at all.  The grid-wide wait moves to the
//     END of the CTA, so that this grid cannot complete before its predecessor has (anything launched after it without
//     the PDL attribute still sees every earlier step finished).  Works unchanged under CUDA-graph replay (nothing
//     about launch order is baked into the launch).
//     Measured (B200, 4 x 2^20 envs round-robin on ONE stream, profiles/exp/r2_step_ring/): 13.4 -> 12.1 us per launch;
//     on 4 parallel graph branches or at 2^24 envs, where (a) has no bubble to lose, the ticket round trip costs 5 %
//     -- the host picks the mode by size.  Also measured there and NOT adopted: a persistent one-CTA-per-SM kernel
//     streaming tiles through a shared-memory ring with cp.async.bulk (12.1 us in the best of 15 configurations, one
//     of which hung), and CTAs that step 2 or 4 tiles (a loop makes ptxas spill the freshly loaded rows; straight-line
//     copies blow the instruction cache: 16 us).
//
// kLog (cartpole_step_logged_kernel, auto-reset only): the thread that resets env i first writes the record of the
// episode that ended -- the xi row before its resample, the state the owner stored, the length and truncated bit the
// owner staged in s_len -- into the episode log.  All of it precedes the tile's release / the end of the grid.
template <typename T, bool kAutoReset, bool kNoisy = false, bool kLean = false>
__global__ void __launch_bounds__(kStepThreads, kNoisy ? (sizeof(T) == 8 ? 2 : 3) : kStepMinCtas<T>) cartpole_step_kernel(const __grid_constant__ StepArgs<T> a)
{
    constexpr bool kLog = false;
    const LogPtrs<T> log = {};
#include "renv_step_body.cuh"
}

template <typename T> struct LoggedStepArgs { StepArgs<T> step; LogPtrs<T> log; };

// The plain auto-reset step plus the episode log (a kernel of its own: the plain one keeps its parameter layout).
template <typename T>
__global__ void __launch_bounds__(kStepThreads, kStepMinCtas<T>) cartpole_step_logged_kernel(const __grid_constant__ LoggedStepArgs<T> args)
{
    constexpr bool kAutoReset = true, kNoisy = false, kLean = false, kLog = true;
    const StepArgs<T> &a = args.step;
    const LogPtrs<T> &log = args.log;
#include "renv_step_body.cuh"
}

// ------------------------------------------------------------------------------------------------
// Reset: RandomCartPoleEnv.reset (+ set_random_task) for masked envs
// ------------------------------------------------------------------------------------------------
template <typename T> struct ResetArgs {
    EnvPtrs<T> env;
    const uint8_t *mask;
    uint64_t tick;
    DrCfg4<T> dr;
    unsigned long long *violations;
};

template <typename T> __global__ void __launch_bounds__(256) cartpole_reset_kernel(const __grid_constant__ ResetArgs<T> a)
{
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= a.env.n) return;
    if (a.mask && !a.mask[i]) return;
    if (a.env.elapsed) a.env.elapsed[i] = 0;
    if (a.env.elapsed16) a.env.elapsed16[i] = 0;
    if (a.env.beyond) a.env.beyond[i] = -1;
    const unsigned viol = reset_env(a.env, a.dr, i, a.tick, a.env.seed);
    if (viol && a.violations) atomicAdd(a.violations, (unsigned long long)viol);
}

// ------------------------------------------------------------------------------------------------
// Fused K-step rollout with in-register state/xi/counters and an in-kernel linear policy
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void atomic_min_f64(double *addr, double v)
{
    unsigned long long *p = reinterpret_cast<unsigned long long *>(addr);
    unsigned long long old = *p;
    while (v < __longlong_as_double((long long)old)) {
        const unsigned long long seen = atomicCAS(p, old, (unsigned long long)__double_as_longlong(v));
        if (seen == old) break;
        old = seen;
    }
}
__device__ __forceinline__ void atomic_max_f64(double *addr, double v)
{
    unsigned long long *p = reinterpret_cast<unsigned long long *>(addr);
    unsigned long long old = *p;
    while (v > __longlong_as_double((long long)old)) {
        const unsigned long long seen = atomicCAS(p, old, (unsigned long long)__double_as_longlong(v));
        if (seen == old) break;
        old = seen;
    }
}

constexpr int kRolloutThreads = 256;

// Episode statistics of one launch: warp shuffle -> shared -> one set of atomics per CTA into the 6 doubles
// [episodes, sum return, sum return^2, min, max, sum length] (the vector the ranks all-gather).
__device__ __forceinline__ void rollout_publish(double *stats, unsigned long long *violations, unsigned episodes,
                                                unsigned sum_len, unsigned sum_r_u, unsigned long long sum_r2_u,
                                                float min_r, float max_r, unsigned viol)
{
    double sum_r = (double)sum_r_u, sum_r2 = (double)sum_r2_u;
    double cnt = (double)episodes, len = (double)sum_len;
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) {
        cnt += __shfl_xor_sync(0xffffffffu, cnt, off);
        len += __shfl_xor_sync(0xffffffffu, len, off);
        sum_r += __shfl_xor_sync(0xffffffffu, sum_r, off);
        sum_r2 += __shfl_xor_sync(0xffffffffu, sum_r2, off);
        min_r = fminf(min_r, __shfl_xor_sync(0xffffffffu, min_r, off));
        max_r = fmaxf(max_r, __shfl_xor_sync(0xffffffffu, max_r, off));
        viol += __shfl_xor_sync(0xffffffffu, viol, off);
    }
    __shared__ double sh[kRolloutThreads / 32][4];
    __shared__ float shm[kRolloutThreads / 32][2];
    __shared__ unsigned shv[kRolloutThreads / 32];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    if (lane == 0) {
        sh[warp][0] = cnt; sh[warp][1] = sum_r; sh[warp][2] = sum_r2; sh[warp][3] = len;
        shm[warp][0] = min_r; shm[warp][1] = max_r; shv[warp] = viol;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        const int nw = blockDim.x >> 5;
        for (int w = 1; w < nw; ++w) {
            cnt += sh[w][0]; sum_r += sh[w][1]; sum_r2 += sh[w][2]; len += sh[w][3];
            min_r = fminf(min_r, shm[w][0]); max_r = fmaxf(max_r, shm[w][1]); viol += shv[w];
        }
        if (cnt > 0.0) {
            atomicAdd(stats + 0, cnt);
            atomicAdd(stats + 1, sum_r);
            atomicAdd(stats + 2, sum_r2);
            atomic_min_f64(stats + 3, (double)min_r);
            atomic_max_f64(stats + 4, (double)max_r);
            atomicAdd(stats + 5, len);
        }
        if (viol && violations) atomicAdd(violations, (unsigned long long)viol);
    }
}

// Statistics of a population launch (cartpole_population_linear_kernel), whose warps may serve two or more members:
// a warp whose lanes all serve one member reduces by shuffles and lane 0 publishes into the member's row; in a warp
// that straddles members every lane with a finished episode publishes into its own member's row.  The six values are
// exact in doubles (integer sums below 2^53, min, max), so the order of the atomics does not change the bits.
__device__ __forceinline__ void population_publish(double *stats, int64_t member, unsigned long long *violations,
                                                   unsigned episodes, unsigned sum_len, unsigned sum_r_u,
                                                   unsigned long long sum_r2_u, float min_r, float max_r, unsigned viol)
{
    double sum_r = (double)sum_r_u, sum_r2 = (double)sum_r2_u;
    double cnt = (double)episodes, len = (double)sum_len;
    const bool shared = __all_sync(0xffffffffu, member == __shfl_sync(0xffffffffu, member, 0));
    if (shared) {
#pragma unroll
        for (int off = 16; off > 0; off >>= 1) {
            cnt += __shfl_xor_sync(0xffffffffu, cnt, off);
            len += __shfl_xor_sync(0xffffffffu, len, off);
            sum_r += __shfl_xor_sync(0xffffffffu, sum_r, off);
            sum_r2 += __shfl_xor_sync(0xffffffffu, sum_r2, off);
            min_r = fminf(min_r, __shfl_xor_sync(0xffffffffu, min_r, off));
            max_r = fmaxf(max_r, __shfl_xor_sync(0xffffffffu, max_r, off));
            viol += __shfl_xor_sync(0xffffffffu, viol, off);
        }
    }
    if (shared && (threadIdx.x & 31) != 0) return;
    if (cnt > 0.0) {
        atomicAdd(stats + 0, cnt);
        atomicAdd(stats + 1, sum_r);
        atomicAdd(stats + 2, sum_r2);
        atomic_min_f64(stats + 3, (double)min_r);
        atomic_max_f64(stats + 4, (double)max_r);
        atomicAdd(stats + 5, len);
    }
    if (viol && violations) atomicAdd(violations, (unsigned long long)viol);
}

template <typename T> struct RolloutArgs {
    EnvPtrs<T> env;
    Policy<T> policy;
    int K, euler, max_steps;
    uint64_t tick;
    DrCfg4<T> dr;
    double *stats;
    unsigned long long *violations;
};

// One env-step of the rollout: policy -> dynamics -> TimeLimit -> (rare) end-of-episode bookkeeping.
// The reset itself is DEFERRED: the lane parks (t.waiting) with the clock tick of the step that ended the
// episode, and the warp executes the ~250-instruction Philox / DR-sampling path once for several parked lanes
// (kResetBatch) instead of once per finished lane with one lane active.  A parked lane simply resumes later and
// runs its remaining steps after the others, so every env still performs exactly K steps with the same
// (seed, id, tick) draws: results are bit-identical to K single-step launches.
struct ActionBits { uint4 r; uint32_t group; };     // an env's 128 action bits for steps 128 g .. 128 g + 127 (random policy)
template <typename T> struct RolloutThread {
    State<T> s; Xi<T> p; Derived<T> d;
    int32_t el; uint32_t new_episodes; bool xi_dirty;
    int remaining;      // steps this lane may still execute now (0 while parked or finished)
    int parked;         // steps left after the pending reset, -1 when not parked
    // Noisy variant only: the observation the policy sees at the next step.  Either the one found in the obs buffer
    // at launch (obs_loaded), or state + std * N(0,I) keyed by the tick that produced the state and `after_reset`
    // (0: a step's observation, 1: a reset's) -- exactly what step() / reset() wrote for that tick.
    State<T> obs0; bool obs_loaded; uint32_t after_reset;
    unsigned long long sum_r2; unsigned sum_r; float min_r, max_r; unsigned episodes, sum_len, viol;
    ActionBits act;     // random policy only: the env's current 128 action bits
    bool refresh;       // ... and: parked for new action bits only, the episode goes on
};

constexpr int kResetBatch = 4;             // parked lanes per warp that trigger a reset pass
constexpr int kStepsPerCheck = 8;          // env-steps between two warp votes
constexpr int kUnrollF64 = 2;
// The fp32 random policy ends an episode every ~25 steps: its own vote period / batch size / unroll.  Measured at
// 2^24 envs x 500 steps (check, batch -> 1e11 env-steps/s): (4,4) 2.48, (8,4) 2.92, (12,4) 3.05, (16,8) 3.11,
// (16,12) 3.08, (20,12) 3.06, (24,12) 2.95, (32,16) 2.61; unroll 1 / 2 / 4 / 8 at (8,4): 2.79 / 2.92 / 2.81 / 2.75.
constexpr int kRandomResetBatch = 8, kRandomStepsPerCheck = 16, kRandomUnroll = 2;

// Bernoulli(1/2) action of env `id` at clock `step` (low 32 bits of the tick): bit (step & 127) of the env's OWN Philox
// block (id, step >> 7) -- the bit random_actions_kernel writes for that env and tick, so a random-policy rollout equals
// K x step(sample_actions()).  One block carries an env's actions for 128 consecutive steps: the fused rollout keeps it
// in registers and draws a new one every 128 env-steps (round 1 keyed the block by (id >> 7, step): every env-step
// re-derived a whole block for one bit, and the random-policy rollout ran at 0.11 of the FMA peak).
__device__ __forceinline__ uint32_t action_bit(const uint4 &r, uint32_t step)
{
    // bit (step & 127) of the 128-bit block x | y << 32 | z << 64 | w << 96, without a branch: two selects pick the
    // 64-bit half, one 64-bit shift the bit (a 4-way word select compiled to a divergent branch tree, ~12 issue slots)
    const bool hi = (step & 64u) != 0u;
    const uint64_t half = (uint64_t)(hi ? r.w : r.y) << 32 | (uint64_t)(hi ? r.z : r.x);
    return (uint32_t)(half >> (step & 63u)) & 1u;
}
template <typename T, bool kEuler, bool kKnownSmall, bool kNoisy = false, bool kRandom = false>
__device__ __forceinline__ void rollout_step(RolloutThread<T> &t, const RolloutArgs<T> &a, const Policy<T> &policy,
                                             int32_t limit, uint64_t id = 0)
{
    int action;
    uint32_t step = 0u;
    if (kRandom) {      // action_space.sample() of the reference's demo loop (test_random_policy.py:26), per env and tick
        step = (uint32_t)a.tick + (uint32_t)(a.K - t.remaining);
        action = (int)action_bit(t.act.r, step);        // t.act always holds the block of step >> 7 (see below)
    } else if (kNoisy) {       // the policy acts on the OBSERVATION of the current state (what step()/reset() returned for it)
        State<T> o = t.obs0;
        if (!t.obs_loaded) {
            T ov[4];
            const uint64_t tick_now = a.tick + (uint64_t)(a.K - t.remaining);
            add_obs_noise(t.s, a.env.noise_std, a.env.seed, id, tick_now - 1, t.after_reset, ov);
            o = State<T>{ ov[0], ov[1], ov[2], ov[3] };
        }
        t.obs_loaded = false; t.after_reset = 0u;
        action = policy_action(policy, o);
    } else {
        action = policy_action(policy, t.s);
    }
    const bool terminated = dynamics<kKnownSmall>(t.s, t.p, t.d, action, kEuler);
    t.el += 1;
    // End of episode: two selects, no branch (some lane of the warp ends an episode on most steps of a short-episode
    // policy, so a branch here is taken by nearly every warp).  The lane sits out with t.el = the episode's length;
    // statistics and the reset itself happen in rollout_reset.
    const bool ended = terminated || t.el >= limit;
    bool park = ended;
    if (kRandom) {
        // The env's 128 action bits run out after this step: the lane parks like one whose episode ended and gets the
        // next block in the warp's reset pass, together with the other parked lanes, instead of running Philox alone
        // inside the step loop (22 % of the warp-steps had such a lane: 10 issue slots per step).
        const bool cross = ((step + 1u) & 127u) == 0u;
        t.refresh = cross && !ended;
        park = ended || cross;
    }
    t.parked = park ? t.remaining - 1 : t.parked;
    t.remaining = park ? 0 : t.remaining - 1;
}

template <typename T, bool kRandom = false>
__device__ __forceinline__ void rollout_reset(RolloutThread<T> &t, const RolloutArgs<T> &a, uint64_t id)
{
    if (!(kRandom && t.refresh)) {
        // the episode that just ended (return == length: the reward is 1.0 on every step, :207-212)
        const float ret = (float)t.el;
        t.episodes += 1; t.sum_len += (unsigned)t.el;
        t.sum_r += (unsigned)t.el; t.sum_r2 += (unsigned long long)t.el * (unsigned)t.el;
        t.min_r = fminf(t.min_r, ret); t.max_r = fmaxf(t.max_r, ret);
        t.new_episodes += 1; t.el = 0;
        // the clock value a single step() would have used for the step that ended it: t.parked steps were left after it
        const uint64_t reset_tick = a.tick + (uint64_t)(a.K - t.parked - 1);
        if (a.dr.dr_type != kDrNone) {
            t.p = Xi<T>{ T(0), T(0), T(0), T(0) };
            t.viol += sample_xi(t.p, a.dr, a.env.seed, id, reset_tick);
            t.d = derive(t.p);
            t.xi_dirty = true;
        }
        init_state(t.s, a.env.seed, id, reset_tick);
        t.after_reset = 1u;
    }
    if (kRandom) {      // the action bits of the step the lane resumes at
        const uint32_t group = ((uint32_t)a.tick + (uint32_t)(a.K - t.parked)) >> 7;
        if (group != t.act.group) {
            t.act.group = group;
            t.act.r = draw_block(a.env.seed, id, (uint64_t)group, kAction, 0);
        }
        t.refresh = false;
    }
    t.remaining = t.parked;
    t.parked = -1;
}

// Keeps a kernel parameter in an ordinary register for the whole loop (nvcc otherwise re-loads it from the
// constant bank through a uniform register on every iteration: 5 extra issue slots per env-step).
__device__ __forceinline__ float pin(float v) { asm volatile("" : "+f"(v)); return v; }
__device__ __forceinline__ double pin(double v) { asm volatile("" : "+d"(v)); return v; }

// Resident CTAs per SM (register cap) of the rollout kernels: 3, and 2 for the fp64 noisy / random-policy ones.
template <typename T> constexpr int rollout_ctas(bool noisy, bool random) { return sizeof(T) == 4 || !(noisy || random) ? 3 : 2; }

// A population launch (renv_cartpole_population_*_f32): P policies, each on the env's n envs from a fresh start.
struct PopulationPtrs {
    const float *policies;      // member p's row: (P, 5) linear w0..w3, b, or (P, kMlpParamFloats) packed MLP parameters
    int64_t total;              // linear kernel: P n, the flat (member, env) index range
    uint32_t ctas;              // MLP kernel: CTAs per member, ceil(n / kMlpThreads)
};

template <typename T, bool kEuler, bool kNoisy = false, bool kRandom = false>
__global__ void __launch_bounds__(kRolloutThreads, rollout_ctas<T>(kNoisy, kRandom))
cartpole_rollout_kernel(const __grid_constant__ RolloutArgs<T> a)
{
    constexpr bool kLog = false, kPop = false;
    const LogPtrs<T> log = {};
    constexpr PopulationPtrs pop = {};
#include "renv_rollout_body.cuh"
}

template <typename T> struct LoggedRolloutArgs { RolloutArgs<T> roll; LogPtrs<T> log; };

// The plain (not Noisy) rollout plus the episode log: fp64, and fp32 under the random policy.
template <typename T, bool kEuler, bool kRandom>
__global__ void __launch_bounds__(kRolloutThreads, rollout_ctas<T>(false, kRandom))
cartpole_rollout_logged_kernel(const __grid_constant__ LoggedRolloutArgs<T> args)
{
    constexpr bool kNoisy = false, kLog = true, kPop = false;
    const RolloutArgs<T> &a = args.roll;
    const LogPtrs<T> &log = args.log;
    constexpr PopulationPtrs pop = {};
#include "renv_rollout_body.cuh"
}

struct PopulationArgs { RolloutArgs<float> roll; PopulationPtrs pop; };     // roll.policy is unused

// P linear policies on the env's n envs, one (member, env) pair per thread over a flat index, so that a population of
// many members with few envs each (ARS / ES: n of 1 to 64) still fills the GPU.  The generic one-env-per-thread body:
// the FFMA2 pair body parks ended envs through the env's buffers, and this kernel writes nothing into the env.
template <bool kEuler>
__global__ void __launch_bounds__(kRolloutThreads, rollout_ctas<float>(false, false))
cartpole_population_linear_kernel(const __grid_constant__ PopulationArgs args)
{
    using T = float;
    constexpr bool kNoisy = false, kRandom = false, kLog = false, kPop = true;
    const RolloutArgs<T> &a = args.roll;
    const LogPtrs<T> log = {};
    const PopulationPtrs &pop = args.pop;
#include "renv_rollout_body.cuh"
}

// ------------------------------------------------------------------------------------------------
// Host path: done / truncated flags cross PCIe as bits (n / 8 bytes instead of n)
// ------------------------------------------------------------------------------------------------
// 4 flag bytes -> 4 bits (bit k set when byte k != 0)
__device__ __forceinline__ uint32_t nibble_of(uint32_t v)
{
    return ((__vcmpne4(v, 0u) & 0x08040201u) * 0x01010101u) >> 24;
}
// Thread w packs flags[32 w .. 32 w + 31] into bits[w]: bit (i & 31) of word i >> 5, i.e. bit (i & 7) of byte i >> 3
// (numpy's bitorder="little").  Flags past n count as 0.
__global__ void __launch_bounds__(256)
pack_flags_kernel(const uint8_t *__restrict__ flags, uint32_t *__restrict__ bits, int64_t n)
{
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t i0 = w * 32;
    if (i0 >= n) return;
    uint32_t out = 0u;
    if (i0 + 32 <= n && (reinterpret_cast<uintptr_t>(flags) & 15u) == 0u) {
        const uint4 a = __ldg(reinterpret_cast<const uint4 *>(flags + i0));
        const uint4 b = __ldg(reinterpret_cast<const uint4 *>(flags + i0) + 1);
        out = nibble_of(a.x) | nibble_of(a.y) << 4 | nibble_of(a.z) << 8 | nibble_of(a.w) << 12 |
              nibble_of(b.x) << 16 | nibble_of(b.y) << 20 | nibble_of(b.z) << 24 | nibble_of(b.w) << 28;
    } else {
        for (int k = 0; k < 32 && i0 + k < n; ++k) out |= (flags[i0 + k] != 0 ? 1u : 0u) << k;
    }
    bits[w] = out;
}

// ------------------------------------------------------------------------------------------------
// RandomEnv.sample_tasks(n) -> (n, dim) row-major, dim <= 32
// ------------------------------------------------------------------------------------------------
constexpr int kSampleThreads = 256;
// Samples per CTA: every thread produces `items` work items whatever `dim` is, so the per-thread set-up (12 parameter
// conversions, ~100 instructions) is amortised: measured at 2^24 x 30 fp32 uniform, 4 / 8 / 16 / 32 items per thread
// give 2.5 / 3.9 / 4.2 / 4.4 TB/s.  The host picks `items` from the problem size (sampler_items) so that small calls
// still spread over all SMs; the kernel only sees the resulting tile.
constexpr int kSamplerItemsMin = 4, kSamplerItemsMax = 32;
template <typename T> __host__ __device__ inline int sampler_log2pad(int dim)
{
    const int blocks_per_sample = (dim + (int)(16 / sizeof(T)) - 1) / (int)(16 / sizeof(T));
    int log2pad = 0;
    while ((1 << log2pad) < blocks_per_sample) ++log2pad;
    return log2pad;
}
template <typename T> inline int sampler_items(int64_t n, int dim)
{
    const int64_t work = n << sampler_log2pad<T>(dim);                 // (sample, block) items incl. padding
    const int64_t per_thread = work / ((int64_t)kSampleThreads * 148 * 8);    // keep >= 8 CTAs per SM in flight
    int items = kSamplerItemsMin;
    while (items < kSamplerItemsMax && items < per_thread) items *= 2;
    return items;
}
template <typename T> __host__ __device__ inline int tile_samples(int dim, int items)
{
    return (kSampleThreads * items) >> sampler_log2pad<T>(dim);
}


// Work item = (sample, dim block of 4 floats / 2 doubles = one Philox call).  Thread t owns dim block
// j = t % jpad (jpad = blocks per sample rounded up to a power of two) for the whole kernel, so its distribution
// parameters are read and converted ONCE into registers and the sample loop is Philox + transform + store, with
// shifts instead of divisions.  Consecutive lanes hold consecutive (sample, block) items = consecutive 16-byte
// chunks of the row-major (n, dim) output, so each warp store instruction covers one contiguous span and no
// shared-memory staging is needed; the store width follows the row alignment (dim % 4 == 0: 128-bit,
// dim even: 64-bit pairs -- e.g. the 30-dim humanoid --, otherwise scalars).
// kStore: 0 = one 128-bit store per block (float: dim % 4 == 0, double: dim even), 1 = float pairs (dim even),
// 2 = scalars.  A template parameter like kDrType: a per-item `switch` on kernel parameters costs an LDC with a
// ~40-cycle scoreboard wait in front of every Philox chain (ncu: short_scoreboard was the top stall).
template <typename T, int kStore> __device__ __forceinline__ void store_block(T *row, const T *v, unsigned valid);
template <> __device__ __forceinline__ void store_block<float, 0>(float *row, const float *v, unsigned)
{
    *reinterpret_cast<float4 *>(row) = make_float4(v[0], v[1], v[2], v[3]);
}
template <> __device__ __forceinline__ void store_block<float, 1>(float *row, const float *v, unsigned valid)
{
    *reinterpret_cast<float2 *>(row) = make_float2(v[0], v[1]);
    if (valid & 4u) *reinterpret_cast<float2 *>(row + 2) = make_float2(v[2], v[3]);
}
template <> __device__ __forceinline__ void store_block<float, 2>(float *row, const float *v, unsigned valid)
{
#pragma unroll
    for (int k = 0; k < 4; ++k)
        if (valid & (1u << k)) row[k] = v[k];
}
template <> __device__ __forceinline__ void store_block<double, 0>(double *row, const double *v, unsigned)
{
    *reinterpret_cast<double2 *>(row) = make_double2(v[0], v[1]);
}
template <> __device__ __forceinline__ void store_block<double, 2>(double *row, const double *v, unsigned valid)
{
    row[0] = v[0];
    if (valid & 2u) row[1] = v[1];
}
template <> __device__ __forceinline__ void store_block<double, 1>(double *row, const double *v, unsigned valid)
{
    store_block<double, 2>(row, v, valid);
}

template <typename T, int kDrType, int kStore>
__global__ void __launch_bounds__(kSampleThreads) dr_sample_kernel(T *__restrict__ out, int64_t n, const DrCfgPrepared<T> cfg,
                                                                   uint64_t seed, uint64_t sample_id0, uint32_t call,
                                                                   unsigned long long *violations, int items)
{
    constexpr int P = Pack<T>::kPerBlock;
    const int dim = cfg.dim;
    const int kTile = tile_samples<T>(dim, items);
    const int blocks_per_sample = (dim + P - 1) / P;
    int log2pad = 0;
    while ((1 << log2pad) < blocks_per_sample) ++log2pad;
    const int j = threadIdx.x & ((1 << log2pad) - 1);
    const int lane_sample = threadIdx.x >> log2pad, samples_per_pass = kSampleThreads >> log2pad;
    const int64_t first = (int64_t)blockIdx.x * kTile;
    const int samples = (int)min((int64_t)kTile, n - first);
    if (j >= blocks_per_sample) return;
    const DimBlock<T> blk = load_dim_block(cfg, j);
    unsigned viol = 0;
    T *const tile = out + (first + lane_sample) * dim + j * P;      // 64-bit once; 32-bit offsets inside the tile
    const int row_step = samples_per_pass * dim;
    const uint64_t id0 = sample_id0 + (uint64_t)(first + lane_sample);
    // (two interleaved Philox chains per thread were tried: no gain, the limit is IMAD.WIDE issue, not latency)
    int sidx = lane_sample, off = 0;
    for (; sidx < samples; sidx += samples_per_pass, off += row_step) {
        T v[P];
        const uint64_t id = id0 + (uint32_t)(sidx - lane_sample);
        const unsigned pending = first_attempt<T>(kDrType, blk, seed, id, call, kTasks, j, v);
        if (kDrType != kDrUniform && pending) viol += redraws<T>(kDrType, blk, seed, id, call, kTasks, j, pending, v);
        store_block<T, kStore>(tile + off, v, blk.valid);
    }
    if (kDrType == kDrGaussian && viol && violations) atomicAdd(violations, (unsigned long long)viol);
}

// The fp32 specialisation of the loop above (the throughput path; the generic kernel stays for fp64 and is what
// this one was derived from -- same work decomposition, same draws, bit-identical output).  The sampler is bound by
// instruction ISSUE, not by HBM (ncu, round 1: ALU pipe 59 %, stalls math-throttle / not-selected / dispatch; Philox
// alone is 20 IMAD.WIDE + 20 LOP3 per 16 output bytes and tops out at 6.8 TB/s), so every instruction removed from
// the per-block loop is throughput:
//   * the Philox counter of a thread's k-th sample differs from its first only in word 0 (the low half of the
//     sample id) as long as the id does not cross a multiple of 2^32, so the loop runs in (at most two) segments with
//     words 1..3 constant: the first round's M1 * c.z and all its XORs with constants, and the second round's
//     M0 * c'.x, are hoisted by the compiler -- 37 instead of 40 Philox instructions and no 64-bit id arithmetic;
//   * the output pointer is advanced instead of re-derived from a 32-bit offset (2 instead of 4 instructions);
//   * the transforms run on packed pairs (renv_dr.cuh: FFMA2 / FMUL2, the same rounding lane for lane);
//   * attempt 0 only answers "did any dim fall below its floor" (4 FSETP); the retry loop of the reference, with
//     its per-dim bookkeeping, is out of line.
constexpr int kSamplerF32Ctas = 2;     // 90-94 registers: round keys, packed constants and parameters all stay resident
// The reference's retry loop for one block whose first attempt left some dim below its floor (random_env.py:158-171,
// 177-190): out of line, so that the per-block loop of the kernel stays Philox + packed transform + store.
struct RedoneBlock { float v0, v1, v2, v3; unsigned viol; };      // returned in registers: no stack traffic in the loop
template <int kDrType>
__device__ __noinline__ RedoneBlock sampler_redo_block(const DrCfgPrepared<float> *cfg, uint64_t seed, uint64_t id,
                                                       uint32_t call, int j)
{
    const DimBlock<float> blk = load_dim_block(*cfg, j);
    float v[4];
    const unsigned pending = first_attempt<float>(kDrType, blk, seed, id, call, kTasks, j, v);
    const unsigned viol = pending ? redraws<float>(kDrType, blk, seed, id, call, kTasks, j, pending, v) : 0u;
    return RedoneBlock{ v[0], v[1], v[2], v[3], viol };
}

template <int kDrType, int kStore>
__global__ void __launch_bounds__(kSampleThreads, kSamplerF32Ctas)
dr_sample_f32_kernel(float *__restrict__ out, int64_t n, const __grid_constant__ DrCfgPrepared<float> cfg, uint64_t seed,
                     const __grid_constant__ PhiloxKeys ks, uint64_t sample_id0, uint32_t call,
                     unsigned long long *violations, int items)
{
    const int dim = cfg.dim;
    const int kTile = tile_samples<float>(dim, items);
    const int blocks_per_sample = (dim + 3) / 4;
    int log2pad = 0;
    while ((1 << log2pad) < blocks_per_sample) ++log2pad;
    const int j = threadIdx.x & ((1 << log2pad) - 1);
    const int lane_sample = threadIdx.x >> log2pad, samples_per_pass = kSampleThreads >> log2pad;
    const int64_t first = (int64_t)blockIdx.x * kTile;
    const int samples = (int)min((int64_t)kTile, n - first);
    if (j >= blocks_per_sample || lane_sample >= samples) return;
    const DimBlockPacked pb = pack_dim_block(load_dim_block(cfg, j));
    // `ks`: the ten round keys, computed on the host -- as kernel parameters they are constant-bank operands of the
    // Philox XORs (computed here they either occupy 20 registers or are re-added inside the loop, 18 instructions)
    unsigned viol = 0;
    float *row = out + (first + lane_sample) * dim + j * 4;
    const int64_t row_step = (int64_t)samples_per_pass * dim;
    const uint64_t id0 = sample_id0 + (uint64_t)(first + lane_sample);
    int todo = (samples - lane_sample + samples_per_pass - 1) / samples_per_pass;      // samples of this thread
    // samples before the low id word wraps (usually all of them)
    const uint64_t to_wrap = (0x100000000ull - (id0 & 0xffffffffull) + (uint64_t)samples_per_pass - 1) / (uint64_t)samples_per_pass;
    uint64_t id = id0;
    while (todo > 0) {
        const int seg = (int)min((uint64_t)todo, id == id0 ? to_wrap : (uint64_t)todo);    // a tile wraps at most once
        // constant words of the segment's counters: (id hi | tick hi, tick lo, purpose | slot)
        const uint32_t c1 = (uint32_t)(id >> 32) & 0xffffu, c2 = call, c3 = ((uint32_t)kTasks << 24) | (uint32_t)j;
        uint32_t c0 = (uint32_t)id;
        auto one_block = [&](uint32_t ctr0, float *dst) {
            const uint4 r = philox4x32_10(make_uint4(ctr0, c1, c2, c3), ks);
            float v[4];
            if (first_attempt_packed<kDrType>(r, pb, v)) {         // rare
                const RedoneBlock b = sampler_redo_block<kDrType>(&cfg, seed, (id & ~0xffffffffull) | ctr0, call, j);
                v[0] = b.v0; v[1] = b.v1; v[2] = b.v2; v[3] = b.v3;
                viol += b.viol;
            }
            store_block<float, kStore>(dst, v, pb.valid);
        };
        int k = seg;
        if (kDrType != kDrUniform) {
            // the transcendental laws are LATENCY-bound (ncu: `wait` 31-36 % of stalls at 2 CTAs/SM: one serial Philox +
            // Horner chain per thread): two samples per iteration give the scheduler two independent chains
            // ... and both in ONE basic block (the rare floor check is taken once, after both transforms): with the
            // check inside each block the compiler emitted block A, its branch, then block B, and the MUFU-heavy transform
            // of A never overlapped the IMAD-heavy Philox of B.  Gaussian 3.51 -> 3.72 TB/s, truncnorm 3.06 -> 3.32.
            // (Drawing the NEXT pair's Philox blocks beside the current pair's transform -- a software pipeline -- was
            // slower: 3.59 / 3.27; 3 CTAs/SM at 80 registers: 3.74 / 3.21.)
#pragma unroll 1
            for (; k >= 2; k -= 2) {
                const uint32_t c0b = c0 + (uint32_t)samples_per_pass;
                const uint4 ra = philox4x32_10(make_uint4(c0, c1, c2, c3), ks);
                const uint4 rb = philox4x32_10(make_uint4(c0b, c1, c2, c3), ks);
                float va[4], vb[4];
                const bool bad_a = first_attempt_packed<kDrType>(ra, pb, va);
                const bool bad_b = first_attempt_packed<kDrType>(rb, pb, vb);
                if (bad_a || bad_b) {                               // rare
                    if (bad_a) {
                        const RedoneBlock b = sampler_redo_block<kDrType>(&cfg, seed, (id & ~0xffffffffull) | c0, call, j);
                        va[0] = b.v0; va[1] = b.v1; va[2] = b.v2; va[3] = b.v3;
                        viol += b.viol;
                    }
                    if (bad_b) {
                        const RedoneBlock b = sampler_redo_block<kDrType>(&cfg, seed, (id & ~0xffffffffull) | c0b, call, j);
                        vb[0] = b.v0; vb[1] = b.v1; vb[2] = b.v2; vb[3] = b.v3;
                        viol += b.viol;
                    }
                }
                store_block<float, kStore>(row, va, pb.valid);
                store_block<float, kStore>(row + row_step, vb, pb.valid);
                c0 += 2u * (uint32_t)samples_per_pass;
                row += 2 * row_step;
            }
        }
#pragma unroll 1
        for (; k > 0; --k) {
            one_block(c0, row);
            c0 += (uint32_t)samples_per_pass;
            row += row_step;
        }
        id += (uint64_t)seg * (uint64_t)samples_per_pass;
        todo -= seg;
    }
    if (kDrType == kDrGaussian && viol && violations) atomicAdd(violations, (unsigned long long)viol);
}

// The fp64 UNIFORM law on the same loop (what RandomEnv.sample_tasks() of the float64 drop-in API runs): one Philox block
// = two doubles = 16 bytes, so the issue budget per byte is that of the fp32 kernel.  numpy's 53-bit recipe
// u = ((hi >> 5) * 2^26 + (lo >> 6)) * 2^-53 is EXACT in every step (27- and 26-bit integers, powers of two), hence
//   * the two int -> double conversions are an OR into the mantissa of 2^52 and one exact DADD each (I2F.F64 is a
//     quarter-rate instruction),
//   * m = fma(a, 2^26, b) is the exact 53-bit integer, and rn(width * u) == rn((width * 2^-53) * m): the product has
//     the same real value, so low + width * u keeps numpy's two roundings with one DMUL and one DADD.
// Bit-identical to dr_sample_kernel<double, kDrUniform> (tests/test_gpu_samplers.py compares both with the oracle).
__device__ __forceinline__ double exact_u32_to_double(uint32_t v)          // v < 2^32: exact
{
    return __dadd_rn(__hiloint2double(0x43300000, (int)v), -4503599627370496.0);
}
template <int kStore>
__global__ void __launch_bounds__(kSampleThreads, 3)
dr_sample_f64_uniform_kernel(double *__restrict__ out, int64_t n, const __grid_constant__ DrCfgPrepared<double> cfg,
                             const __grid_constant__ PhiloxKeys ks, uint64_t sample_id0, uint32_t call, int items)
{
    const int dim = cfg.dim;
    const int kTile = tile_samples<double>(dim, items);
    const int blocks_per_sample = (dim + 1) / 2;
    int log2pad = 0;
    while ((1 << log2pad) < blocks_per_sample) ++log2pad;
    const int j = threadIdx.x & ((1 << log2pad) - 1);
    const int lane_sample = threadIdx.x >> log2pad, samples_per_pass = kSampleThreads >> log2pad;
    const int64_t first = (int64_t)blockIdx.x * kTile;
    const int samples = (int)min((int64_t)kTile, n - first);
    if (j >= blocks_per_sample || lane_sample >= samples) return;
    const DimBlock<double> blk = load_dim_block(cfg, j);
    const double w0 = blk.b[0] * (1.0 / 9007199254740992.0), w1 = blk.b[1] * (1.0 / 9007199254740992.0);   // exact
    double *row = out + (first + lane_sample) * dim + j * 2;
    const int64_t row_step = (int64_t)samples_per_pass * dim;
    const uint64_t id0 = sample_id0 + (uint64_t)(first + lane_sample);
    int todo = (samples - lane_sample + samples_per_pass - 1) / samples_per_pass;
    const uint64_t to_wrap = (0x100000000ull - (id0 & 0xffffffffull) + (uint64_t)samples_per_pass - 1) / (uint64_t)samples_per_pass;
    uint64_t id = id0;
    while (todo > 0) {
        const int seg = (int)min((uint64_t)todo, id == id0 ? to_wrap : (uint64_t)todo);    // a tile wraps at most once
        const uint32_t c1 = (uint32_t)(id >> 32) & 0xffffu, c2 = call, c3 = ((uint32_t)kTasks << 24) | (uint32_t)j;
        uint32_t c0 = (uint32_t)id;
#pragma unroll 1
        for (int k = seg; k > 0; --k) {
            const uint4 r = philox4x32_10(make_uint4(c0, c1, c2, c3), ks);
            const double m0 = fma(exact_u32_to_double(r.x >> 5), 67108864.0, exact_u32_to_double(r.y >> 6));
            const double m1 = fma(exact_u32_to_double(r.z >> 5), 67108864.0, exact_u32_to_double(r.w >> 6));
            double v[2] = { __dadd_rn(blk.a[0], __dmul_rn(w0, m0)), __dadd_rn(blk.a[1], __dmul_rn(w1, m1)) };
            store_block<double, kStore>(row, v, blk.valid);
            c0 += (uint32_t)samples_per_pass;
            row += row_step;
        }
        id += (uint64_t)seg * (uint64_t)samples_per_pass;
        todo -= seg;
    }
}

// ------------------------------------------------------------------------------------------------
// sample_tasks(n) for dr_type 'fullgaussian' (random_env.py:192-198): x = mean + F z, clip [0,4], denormalise
// ------------------------------------------------------------------------------------------------
// A batched dim x dim mat-vec: 2 dim^2 FLOPs per sample against dim * sizeof(T) output bytes -- FMA-bound for the
// 30-dim humanoid.  One thread = one sample with all (padded) 32 outputs as register accumulators; z is produced
// one Philox block at a time and never stored.  The factor arrives TRANSPOSED and zero-padded to 32 x 32 in the
// kernel parameter block (constant bank), and the k loop is fully unrolled, so every coefficient is an immediate
// constant-bank operand of its FMA: no load instruction at all in the inner product.
//   v1: one output element per thread, two LDS per FMA            11.6 ms for 2^24 x 30 fp32
//   v2: register accumulators, factor broadcast from shared memory   2.2 ms (LSU-bound: an LDS.128 broadcast still
//       costs 4 wavefronts, 256 of them per sample)
//   v3: factor as constant-bank operands                             see DESIGN.md
// Summation order (k ascending, FMA) is the same in all three, so the values never changed.  Rows are staged per
// warp in shared memory and written as 128-bit chunks.
template <typename T> struct FullGaussCfg {
    int dim;
    T mean[32], lo[32], hi[32];
    T ft[32 * 32];               // ft[k * 32 + d] = F[d][k] (F F^T = cov), zero beyond dim: 4 KB fp32 / 8 KB fp64
};
constexpr int kFullGaussThreads = 128, kFullGaussCtas = 4;

// D = dim rounded up to {4, 8, 16, 32}: accumulators and unrolled loops are sized for it (a 4-dim cart-pole sample is
// 16 FMAs, not 1024).
template <typename T, int D>
__global__ void __launch_bounds__(kFullGaussThreads, kFullGaussCtas)
dr_sample_fullgaussian_kernel(T *__restrict__ out, int64_t n, const __grid_constant__ FullGaussCfg<T> cfg, uint64_t seed,
                              uint64_t sample_id0, uint32_t call)
{
    constexpr int P = Pack<T>::kPerBlock;
    constexpr int W = 16 / (int)sizeof(T);                      // elements per 128-bit access
    __shared__ __align__(16) T stage[kFullGaussThreads * D];    // per warp: 32 rows of `dim` values, contiguous
    const int dim = cfg.dim;
    const int64_t i = (int64_t)blockIdx.x * kFullGaussThreads + threadIdx.x;
    const uint64_t id = sample_id0 + (uint64_t)i;
    T x[D];
#pragma unroll
    for (int d = 0; d < D; ++d) x[d] = cfg.mean[d];             // zero beyond dim (host)
    if (i < n) {
#pragma unroll
        for (int j = 0; j < D / P; ++j) {
            if (j * P < dim) {                                  // uniform branch; rows k >= dim of ft are zero anyway
                T z[P];
                Num<T>::normals(draw_block(seed, id, call, kTasks, (uint32_t)j), z);
#pragma unroll
                for (int kk = 0; kk < P; ++kk)
#pragma unroll
                    for (int d = 0; d < D; ++d)
                        x[d] = Num<T>::affine(cfg.ft[(j * P + kk) * 32 + d], z[kk], x[d]);
            }
        }
    }
    // clip, denormalise, stage the row
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    T *tile = stage + warp * 32 * D;
#pragma unroll
    for (int d = 0; d < D; ++d)
        if (d < dim) tile[lane * dim + d] = denormalize(x[d], cfg.lo[d], cfg.hi[d]);
    __syncwarp();
    const int64_t warp_first = (int64_t)blockIdx.x * kFullGaussThreads + warp * 32;
    const int rows = (int)max((int64_t)0, min((int64_t)32, n - warp_first));
    const int total = rows * dim;
    T *dst = out + warp_first * dim;                            // 32 * dim * sizeof(T) is a multiple of 128 bytes
    const int nvec = total / W;
    for (int q = lane; q < nvec; q += 32)
        reinterpret_cast<uint4 *>(dst)[q] = reinterpret_cast<const uint4 *>(tile)[q];
    for (int q = nvec * W + lane; q < total; q += 32) dst[q] = tile[q];
}

// ------------------------------------------------------------------------------------------------
// action_space.sample() for every env: Bernoulli(1/2) bits
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) random_actions_kernel(uint8_t *__restrict__ action, int64_t n, uint64_t env_id0,
                                                             uint64_t seed, uint32_t step)
{
    const int64_t i0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) * 4;
    if (i0 >= n) return;
    uint32_t word = 0;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
        const uint64_t e = env_id0 + (uint64_t)(i0 + k);
        const uint4 r = draw_block(seed, e, (uint64_t)(step >> 7), kAction, 0);
        word |= action_bit(r, step) << (8 * k);
    }
    if (i0 + 4 <= n) {
        *reinterpret_cast<uint32_t *>(action + i0) = word;
    } else {
        for (int k = 0; k < 4 && i0 + k < n; ++k) action[i0 + k] = (uint8_t)((word >> (8 * k)) & 1u);
    }
}

}  // namespace renv
