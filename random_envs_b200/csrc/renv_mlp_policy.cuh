// A trained MLP policy inside the env kernels (include/renv.h renv_mlp_policy):
//
//     Linear(4, 64) -> act -> Linear(64, 64) -> act -> Linear(64, 2),  a = argmax(l0, l1)  (a tie gives 0),
//
// act = tanh or ReLU, narrower nets zero-padded to 64 units on the host (exact: act(0) = 0).  fp32 envs only.
//
// mlp_logits() evaluates the policy for the 32 envs of a warp (one env per lane) and is the ONE implementation all four
// MLP kernels (policy_actions, policy_logp, rollout, collect) call, so that a fused rollout equals K x
// {policy_actions; step} bit for bit by construction: the same instructions, the same head / tail split, the same
// summation order.  Every floating-point operation is an explicit intrinsic, so no kernel can contract it differently.
// mlp_pick() does the same for the sampled action and its log-probability (policy_logp and collect).
//
// Layer 2 (64 x 64, 8,192 of the ~9,000 FLOPs of an env-step) runs on the tensor cores as mma.sync m16n8k8 TF32
// (HMMA.1688.F32.TF32): the warp's 32 envs are two M = 16 row tiles, the 64 outputs eight N = 8 column tiles, the 64
// inputs eight K = 8 steps.  Operands are split into a TF32 head and tail, x = hi + lo, and every product is formed
// as  lo.hi + hi.lo + hi.hi  ("3xTF32": the dropped lo.lo term is ~2^-22 relative) with fp32 accumulation -- fp32-class
// logits; a single TF32 pass misses the 1e-5 accuracy contract by 4-40x (DESIGN.md section 4.9).
//   * Layer 1 (K = 4) is computed straight into the A fragments: a lane needs rows g, g + 8, g + 16, g + 24 (g = lane / 4)
//     and, per K-step, units 8 j + t and 8 j + t + 4 (t = lane % 4) -- 64 activations per lane, each computed once
//     per warp, so the warp does exactly the per-env work.  The four rows' states arrive by shuffles.
//   * W2 is split once per CTA into shared memory, already in B-fragment order: one conflict-free 128-bit load per
//     (K-step, N-tile) gives a lane {hi(k), hi(k + 4), lo(k), lo(k + 4)}.
//   * Layer 3 (N = 2) runs on the C fragments: a lane holds 16 columns of 4 rows, the four lanes of a quad add their
//     partial sums by a butterfly (commutative: every lane gets the same bits) and one more shuffle hands each env's
//     logits to the lane that owns it.
// mma.sync is warp-collective: all 32 lanes execute it; lanes without an env feed a zero state and discard the result.
#pragma once
#include "renv_kernels.cuh"

namespace renv {

constexpr int kMlpHidden = 64;
constexpr int kMlpOffW1 = 0, kMlpOffB1 = 256, kMlpOffW2 = 320, kMlpOffB2 = 4416, kMlpOffW3 = 4480, kMlpOffB3 = 4608;
constexpr int kMlpParamFloats = 4612;     // 4610 rounded up to a multiple of 4 (include/renv.h RENV_MLP_PARAM_FLOATS)
enum MlpAct : int { kMlpTanh = 0, kMlpRelu = 1 };

constexpr int kMlpThreads = 128;
constexpr int kMlpCtas = 4;              // policy_actions: 128 registers, 16 warps per SM
constexpr int kMlpRolloutCtas = 3;       // the rollout keeps its env, task and statistics beside the policy: ~148 registers
                                         // (at 4 CTAs = 128 registers it spills)

// The parameters as the fragments want them (filled by mlp_load_params; ~34 KB).
struct __align__(16) MlpSmem {
    float4 w2[8 * 8 * 32];       // [K-step j][N-tile nt][lane]: W2[8 nt + g][8 j + t], [.. + 4] head, then the same tail
    float4 w1[kMlpHidden];       // W1 rows
    float b1[kMlpHidden];
    float2 b2[8 * 4];            // [nt][t]: b2[8 nt + 2 t], b2[8 nt + 2 t + 1]  (the columns of a lane's C fragment)
    float4 w3[8 * 4];            // [nt][t]: W3[0][c], W3[0][c + 1], W3[1][c], W3[1][c + 1],  c = 8 nt + 2 t
    float b3[2];
};

__device__ __forceinline__ float tf32_head(float x) { return __uint_as_float(__float_as_uint(x) & 0xffffe000u); }

// Cooperative load of the packed parameters (all threads of the CTA; ends with a barrier).
__device__ __forceinline__ void mlp_load_params(MlpSmem &sm, const float *__restrict__ prm)
{
    for (int e = threadIdx.x; e < kMlpHidden * kMlpHidden; e += blockDim.x) {
        const int n = e >> 6, k = e & 63;                       // W2[n][k] is B[k][n]
        const float w = prm[kMlpOffW2 + e];
        const int j = k >> 3, t = k & 3, which = (k >> 2) & 1, nt = n >> 3, g = n & 7;
        float *slot = reinterpret_cast<float *>(&sm.w2[(j * 8 + nt) * 32 + 4 * g + t]);
        const float hi = tf32_head(w);
        slot[which] = hi;
        slot[2 + which] = __fsub_rn(w, hi);                     // exact
    }
    for (int u = threadIdx.x; u < kMlpHidden; u += blockDim.x) {
        sm.w1[u] = reinterpret_cast<const float4 *>(prm + kMlpOffW1)[u];
        sm.b1[u] = prm[kMlpOffB1 + u];
    }
    for (int q = threadIdx.x; q < 32; q += blockDim.x) {
        const int c = 8 * (q >> 2) + 2 * (q & 3);
        sm.b2[q] = make_float2(prm[kMlpOffB2 + c], prm[kMlpOffB2 + c + 1]);
        sm.w3[q] = make_float4(prm[kMlpOffW3 + c], prm[kMlpOffW3 + c + 1], prm[kMlpOffW3 + 64 + c], prm[kMlpOffW3 + 64 + c + 1]);
    }
    if (threadIdx.x < 2) sm.b3[threadIdx.x] = prm[kMlpOffB3 + threadIdx.x];
    __syncthreads();
}

template <int kAct> __device__ __forceinline__ float mlp_act(float x)
{
    return kAct == kMlpTanh ? tanhf(x) : fmaxf(x, 0.0f);      // tanhf: the accurate library tanh (<= 2 ulp), not tanh.approx
}

// D += A B on the tensor cores, m16n8k8, TF32 operands, fp32 accumulation.
__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1)
{
    asm("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0, %1, %2, %3}, {%4, %5, %6, %7}, {%8, %9}, {%0, %1, %2, %3};"
        : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

// Logits of this lane's env (state s) for all 32 lanes of the warp.  Warp-collective: every lane of the warp calls it,
// converged; the result does not depend on the other lanes' states.
template <int kAct>
__device__ __forceinline__ void mlp_logits(const MlpSmem &sm, const State<float> &s, float &l0, float &l1)
{
    const int lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
    float v0 = 0.0f, v1 = 0.0f;  // layer 3 of row g + 8 t, the row this lane hands on (see the end)
    // (a rolled loop: unrolled, the compiler keeps tile 0's 64 shared-memory B fragments live for tile 1)
#pragma unroll 1
    for (int m = 0; m < 2; ++m) {               // row tile m: rows 16 m + g (fragment rows g) and 16 m + g + 8 (g + 8)
        float r0[2], r1[2], r2[2], r3[2];
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int row = 16 * m + 8 * h + g;
            r0[h] = __shfl_sync(0xffffffffu, s.x, row);
            r1[h] = __shfl_sync(0xffffffffu, s.x_dot, row);
            r2[h] = __shfl_sync(0xffffffffu, s.theta, row);
            r3[h] = __shfl_sync(0xffffffffu, s.theta_dot, row);
        }
        float acc[8][4];
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            const float2 b = sm.b2[nt * 4 + t];
            acc[nt][0] = b.x; acc[nt][1] = b.y; acc[nt][2] = b.x; acc[nt][3] = b.y;
        }
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            // layer 1 into the A fragment of K-step j: a0 (g, t), a1 (g + 8, t), a2 (g, t + 4), a3 (g + 8, t + 4)
            uint32_t ahi[4], alo[4];
#pragma unroll
            for (int c = 0; c < 2; ++c) {
                const int u = 8 * j + t + 4 * c;
                const float4 w = sm.w1[u];
                const float bu = sm.b1[u];
#pragma unroll
                for (int h = 0; h < 2; ++h) {
                    const float pre = fmaf(w.w, r3[h], fmaf(w.z, r2[h], fmaf(w.y, r1[h], fmaf(w.x, r0[h], bu))));
                    const float x = mlp_act<kAct>(pre);
                    const float hi = tf32_head(x);
                    ahi[h + 2 * c] = __float_as_uint(hi);
                    alo[h + 2 * c] = __float_as_uint(__fsub_rn(x, hi));
                }
            }
#pragma unroll
            for (int nt = 0; nt < 8; ++nt) {
                const float4 b = sm.w2[(j * 8 + nt) * 32 + lane];
                const uint32_t bh0 = __float_as_uint(b.x), bh1 = __float_as_uint(b.y);
                mma_tf32(acc[nt], alo, bh0, bh1);
                mma_tf32(acc[nt], ahi, __float_as_uint(b.z), __float_as_uint(b.w));
                mma_tf32(acc[nt], ahi, bh0, bh1);
            }
        }
        // layer 3 on the C fragment: c0 (g, 2t), c1 (g, 2t + 1), c2 (g + 8, 2t), c3 (g + 8, 2t + 1) of N-tile nt
        float p0[2] = { 0.0f, 0.0f }, p1[2] = { 0.0f, 0.0f };
#pragma unroll
        for (int nt = 0; nt < 8; ++nt) {
            const float4 w = sm.w3[nt * 4 + t];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const float h0 = mlp_act<kAct>(acc[nt][2 * h]), h1 = mlp_act<kAct>(acc[nt][2 * h + 1]);
                p0[h] = fmaf(w.y, h1, fmaf(w.x, h0, p0[h]));
                p1[h] = fmaf(w.w, h1, fmaf(w.z, h0, p1[h]));
            }
        }
        // the four lanes of a quad add their partial sums (a butterfly: every lane gets the same bits) ...
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            p0[h] = __fadd_rn(p0[h], __shfl_xor_sync(0xffffffffu, p0[h], 1));
            p1[h] = __fadd_rn(p1[h], __shfl_xor_sync(0xffffffffu, p1[h], 1));
            p0[h] = __fadd_rn(p0[h], __shfl_xor_sync(0xffffffffu, p0[h], 2));
            p1[h] = __fadd_rn(p1[h], __shfl_xor_sync(0xffffffffu, p1[h], 2));
        }
        // ... and lane 4 g + t keeps row g + 8 t = 16 m + 8 h + g, i.e. t = 2 m + h
        v0 = t == 2 * m ? p0[0] : t == 2 * m + 1 ? p0[1] : v0;
        v1 = t == 2 * m ? p1[0] : t == 2 * m + 1 ? p1[1] : v1;
    }
    // lane L receives row L from lane 4 (L % 8) + L / 8
    const int src = 4 * (lane & 7) + (lane >> 3);
    l0 = __fadd_rn(__shfl_sync(0xffffffffu, v0, src), sm.b3[0]);
    l1 = __fadd_rn(__shfl_sync(0xffffffffu, v1, src), sm.b3[1]);
}

// argmax(l0, l1) with torch.argmax's tie rule (the first index wins)
__device__ __forceinline__ int mlp_action(float l0, float l1) { return l1 > l0 ? 1 : 0; }

// The action of the softmax policy over (l0, l1) and its log-probability, for env `id` stepping at `tick`: the ONE
// implementation both cartpole_policy_logp_mlp_kernel and cartpole_collect_mlp_kernel call.  With d = l1 - l0:
//   sample: a = [u < sigmoid(d)], u = u01 of word x of block (seed, id, tick, purpose 5, slot 0) (include/renv.h);
//   greedy: a = mlp_action(l0, l1);
//   logp = log sigmoid(d) for a = 1, log sigmoid(-d) for a = 0, as -softplus(-/+d) = -(max(z, 0) + log1p(exp(-|d|))).
// `sample` is warp-uniform in both kernels: the greedy path skips the Philox block.
__device__ __forceinline__ int mlp_pick(float l0, float l1, bool sample, uint64_t seed, uint64_t id, uint64_t tick, float &logp)
{
    const float dl = __fsub_rn(l1, l0);
    int action;
    if (sample) {
        const float u = u01(draw_block(seed, id, tick, kPolicySample, 0).x);
        action = u < __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-dl))) ? 1 : 0;
    } else {
        action = mlp_action(l0, l1);
    }
    const float z = action ? -dl : dl;
    logp = -__fadd_rn(fmaxf(z, 0.0f), log1pf(expf(-fabsf(dl))));
    return action;
}

// Per-step trajectory record of cartpole_collect_mlp_kernel (include/renv.h renv_trajectory): row k * ld + i of each
// field holds step k of env i.  logp, truncated and final_obs may be nullptr.
struct MlpTrajPtrs {
    float *obs;               // (capacity, ld, 4) rows: the observation the action was chosen from
    uint8_t *action, *done;
    float *logp;
    uint8_t *truncated;
    float *final_obs;         // (capacity, ld, 4) rows: the state after the step, written where done
};

// ------------------------------------------------------------------------------------------------
// policy_actions: action[i] (and the logits) for every env, from the env's SoA state
// ------------------------------------------------------------------------------------------------
struct MlpActionArgs {
    const float *state; int64_t n, ld;
    const float *params;
    uint8_t *action;
    float *logits;            // (2, ld) or nullptr
};

// Persistent CTAs (one wave): the parameters are staged once per CTA, not once per 256 envs.
template <int kAct>
__global__ void __launch_bounds__(kMlpThreads, kMlpCtas)
cartpole_policy_actions_mlp_kernel(const __grid_constant__ MlpActionArgs a)
{
    __shared__ MlpSmem sm;
    mlp_load_params(sm, a.params);
    const int64_t ld = a.ld;
    for (int64_t base = (int64_t)blockIdx.x * kMlpThreads; base < a.n; base += (int64_t)gridDim.x * kMlpThreads) {
        const int64_t i = base + threadIdx.x;
        if (base + (threadIdx.x & ~31) >= a.n) break;           // the whole warp is past n (warp-uniform)
        const bool live = i < a.n;
        const State<float> s = live ? State<float>{ a.state[i], a.state[ld + i], a.state[2 * ld + i], a.state[3 * ld + i] }
                                    : State<float>{ 0.0f, 0.0f, 0.0f, 0.0f };
        float l0, l1;
        mlp_logits<kAct>(sm, s, l0, l1);
        if (live) {
            a.action[i] = (uint8_t)mlp_action(l0, l1);
            if (a.logits) { a.logits[i] = l0; a.logits[ld + i] = l1; }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// policy_logp: the sampled (or greedy) action and its log-probability at one tick -- the step-loop twin of collect
// ------------------------------------------------------------------------------------------------
struct MlpLogpArgs {
    MlpActionArgs act;        // state, n, ld, params, action, logits (nullptr: not written)
    float *logp;              // (ld) or nullptr
    uint64_t env_id0, seed, tick;
    int sample;               // 0: argmax, 1: a ~ softmax(l0, l1)
};

// 3 CTAs per SM as the rollout: at 4 (128 registers) the Philox block and log1p beside mlp_logits spill 16 bytes (Tanh).
template <int kAct>
__global__ void __launch_bounds__(kMlpThreads, kMlpRolloutCtas)
cartpole_policy_logp_mlp_kernel(const __grid_constant__ MlpLogpArgs args)
{
    __shared__ MlpSmem sm;
    const MlpActionArgs &a = args.act;
    mlp_load_params(sm, a.params);
    const int64_t ld = a.ld;
    const bool sample = args.sample != 0;
    for (int64_t base = (int64_t)blockIdx.x * kMlpThreads; base < a.n; base += (int64_t)gridDim.x * kMlpThreads) {
        const int64_t i = base + threadIdx.x;
        if (base + (threadIdx.x & ~31) >= a.n) break;           // the whole warp is past n (warp-uniform)
        const bool live = i < a.n;
        const State<float> s = live ? State<float>{ a.state[i], a.state[ld + i], a.state[2 * ld + i], a.state[3 * ld + i] }
                                    : State<float>{ 0.0f, 0.0f, 0.0f, 0.0f };
        float l0, l1;
        mlp_logits<kAct>(sm, s, l0, l1);
        if (live) {
            float logp;
            a.action[i] = (uint8_t)mlp_pick(l0, l1, sample, args.seed, args.env_id0 + (uint64_t)i, args.tick, logp);
            if (args.logp) args.logp[i] = logp;
            if (a.logits) { a.logits[i] = l0; a.logits[ld + i] = l1; }
        }
    }
}

// ------------------------------------------------------------------------------------------------
// Fused K-step rollout under the MLP policy
// ------------------------------------------------------------------------------------------------
struct MlpRolloutArgs {
    RolloutArgs<float> roll;   // roll.policy is unused
    const float *params;
    LogPtrs<float> log;        // read only by the kLog instance
};

// One env per thread, all lanes of a warp in lockstep (mma.sync is collective): a lane whose episode ends resets
// INLINE at the tick of that step -- the reset (~250 instructions) is small next to the policy (1,300-3,100 per warp), so
// the parking and batched resets of the linear rollout (section 4.2) would buy nothing here.  Every draw is keyed by
// (seed, global env id, tick) exactly as in cartpole_step_kernel, and the episode bookkeeping is that kernel's, so the
// launch equals K x {renv_cartpole_policy_actions_mlp_f32; renv_cartpole_step_f32 (auto-reset)} bit for bit.
template <int kAct, bool kEuler, bool kLog>
__global__ void __launch_bounds__(kMlpThreads, kMlpRolloutCtas)
cartpole_rollout_mlp_kernel(const __grid_constant__ MlpRolloutArgs args)
{
    constexpr bool kCollect = false, kPop = false;
    constexpr MlpTrajPtrs traj = {};
    constexpr bool sample = false;
    constexpr PopulationPtrs pop = {};
#include "renv_mlp_rollout_body.cuh"
}

// ------------------------------------------------------------------------------------------------
// Fused K-step trajectory collection: the rollout above plus the sampled action, its log-probability and the per-step
// record a policy-gradient learner needs
// ------------------------------------------------------------------------------------------------
struct MlpCollectArgs {
    RolloutArgs<float> roll;   // roll.policy is unused
    const float *params;
    LogPtrs<float> log;        // read only by the kLog instance
    MlpTrajPtrs traj;
    int sample;                // 0: argmax, 1: a ~ softmax(l0, l1)  (warp-uniform)
};

// Step k of env i stores obs, action and logp before the dynamics, done and truncated after them, and final_obs where
// the episode ended, before its reset; the env, the statistics and the log are handled exactly as in
// cartpole_rollout_mlp_kernel (the same body).  The action comes from mlp_pick, which policy_logp also calls, so the
// launch equals K x {record obs; renv_cartpole_policy_logp_mlp_f32; renv_cartpole_step_f32 (auto-reset)} bit for bit.
// Greed / sampling is a runtime argument: one instance per (activation, integrator, log) as for the rollout.
template <int kAct, bool kEuler, bool kLog>
__global__ void __launch_bounds__(kMlpThreads, kMlpRolloutCtas)
cartpole_collect_mlp_kernel(const __grid_constant__ MlpCollectArgs args)
{
    constexpr bool kCollect = true, kPop = false;
    const MlpTrajPtrs &traj = args.traj;
    const bool sample = args.sample != 0;
    constexpr PopulationPtrs pop = {};
#include "renv_mlp_rollout_body.cuh"
}

// ------------------------------------------------------------------------------------------------
// Population evaluation: P MLP policies (one activation), each on the env's n envs from a fresh start
// ------------------------------------------------------------------------------------------------
struct MlpPopulationArgs {
    MlpRolloutArgs mlp;        // mlp.roll.policy, mlp.params and mlp.log are unused
    PopulationPtrs pop;        // pop.policies: (P, kMlpParamFloats) rows; pop.ctas = ceil(n / kMlpThreads)
};

// The rollout body with one member per CTA: the CTA stages its member's parameter row and runs ceil(n / 128) of its
// envs.  P x ceil(n / 128) CTAs on a 1-D grid; lanes past n idle, so a launch keeps n / (128 ceil(n / 128)) of its
// lanes busy (1 at n = 128 k, 0.5 at n = 64, 1 / 128 at n = 1).
template <int kAct, bool kEuler>
__global__ void __launch_bounds__(kMlpThreads, kMlpRolloutCtas)
cartpole_population_mlp_kernel(const __grid_constant__ MlpPopulationArgs pa)
{
    constexpr bool kLog = false, kCollect = false, kPop = true;
    constexpr MlpTrajPtrs traj = {};
    constexpr bool sample = false;
    const MlpRolloutArgs &args = pa.mlp;
    const PopulationPtrs &pop = pa.pop;
#include "renv_mlp_rollout_body.cuh"
}

}  // namespace renv
