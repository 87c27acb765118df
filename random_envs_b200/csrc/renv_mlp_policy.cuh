// A trained MLP policy inside the env kernels (include/renv.h renv_mlp_policy):
//
//     Linear(4, 64) -> act -> Linear(64, 64) -> act -> Linear(64, 2),  a = argmax(l0, l1)  (a tie gives 0),
//
// act = tanh or ReLU, narrower nets zero-padded to 64 units on the host (exact: act(0) = 0).  fp32 envs only.
//
// mlp_logits() evaluates the policy for the 32 envs of a warp (one env per lane) and is the ONE implementation both
// cartpole_policy_actions_mlp_kernel and cartpole_rollout_mlp_kernel call, so that a fused rollout equals K x
// {policy_actions; step} bit for bit by construction: the same instructions, the same head / tail split, the same
// summation order.  Every floating-point operation is an explicit intrinsic, so no kernel can contract it differently.
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
#ifndef RENV_MLP_EXP_PASSES
#define RENV_MLP_EXP_PASSES 3    // experiment knob (DESIGN.md section 4.9): 1 = head x head only, a third of the HMMAs
#endif
#ifndef RENV_MLP_CTAS
#define RENV_MLP_CTAS 4          // policy_actions: 128 registers, 16 warps per SM
#endif
#ifndef RENV_MLP_ROLLOUT_CTAS
#define RENV_MLP_ROLLOUT_CTAS 3  // the rollout keeps its env, task and statistics beside the policy: ~148 registers
                                 // (at 4 CTAs = 128 registers it spills)
#endif

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
#if RENV_MLP_EXP_PASSES == 3
                mma_tf32(acc[nt], alo, bh0, bh1);
                mma_tf32(acc[nt], ahi, __float_as_uint(b.z), __float_as_uint(b.w));
#endif
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
__global__ void __launch_bounds__(kMlpThreads, RENV_MLP_CTAS)
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
__global__ void __launch_bounds__(kMlpThreads, RENV_MLP_ROLLOUT_CTAS)
cartpole_rollout_mlp_kernel(const __grid_constant__ MlpRolloutArgs args)
{
    __shared__ MlpSmem sm;
    mlp_load_params(sm, args.params);
    const RolloutArgs<float> &a = args.roll;
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t ld = a.env.ld;
    const bool live = i < a.env.n;
    const int64_t il = live ? i : 0;
    const uint64_t id = a.env.env_id0 + (uint64_t)il;

    State<float> s = live ? State<float>{ a.env.state[i], a.env.state[ld + i], a.env.state[2 * ld + i], a.env.state[3 * ld + i] }
                          : State<float>{ 0.0f, 0.0f, 0.0f, 0.0f };      // lanes past n feed zero rows
    Xi<float> p = load_xi(a.env.xi, il);
    Derived<float> d = derive(p);
    int32_t el = a.env.elapsed[il];
    uint32_t log_count = kLog ? (uint32_t)args.log.count[il] : 0u;
    unsigned episodes = 0, sum_len = 0, viol = 0;         // return == length (:207-212): sum_len is also sum R
    unsigned long long sum_r2 = 0;
    float min_r = __int_as_float(0x7f800000), max_r = __int_as_float(0xff800000);
    bool xi_dirty = false;

    if (__any_sync(0xffffffffu, live)) {                        // warp-uniform: a warp entirely past n only publishes
        for (int k = 0; k < a.K; ++k) {
            float l0, l1;
            mlp_logits<kAct>(sm, s, l0, l1);
            if (live) {
                const int action = mlp_action(l0, l1);
                // step 0 may start from an injected state at any angle; from step 1 on |theta| <= 0.2095 holds at
                // every step start (an env beyond the threshold was just reset): the same bits without the range check
                const bool terminated = k == 0 ? dynamics<false>(s, p, d, action, kEuler)
                                               : dynamics<true>(s, p, d, action, kEuler);
                el += 1;                                                   // TimeLimit.step
                if (terminated || (a.max_steps > 0 && el >= a.max_steps)) {
                    const uint64_t tick = a.tick + (uint64_t)k;
                    const float ret = (float)el;
                    episodes += 1; sum_len += (unsigned)el;
                    sum_r2 += (unsigned long long)el * (unsigned)el;
                    min_r = fminf(min_r, ret); max_r = fmaxf(max_r, ret);
                    if (kLog) {
                        log_episode(args.log, ld, i, log_count, p, s, el, !terminated, tick);
                        log_count += 1u;
                    }
                    el = 0;
                    if (a.dr.dr_type != kDrNone) {                         // reset_env: set_random_task, then reset
                        p = Xi<float>{ 0.0f, 0.0f, 0.0f, 0.0f };
                        viol += sample_xi(p, a.dr, a.env.seed, id, tick);
                        d = derive(p);
                        xi_dirty = true;
                    }
                    init_state(s, a.env.seed, id, tick);
                }
            }
            __syncwarp();
        }
    }

    if (live) {
        a.env.state[i] = s.x; a.env.state[ld + i] = s.x_dot; a.env.state[2 * ld + i] = s.theta; a.env.state[3 * ld + i] = s.theta_dot;
        if (xi_dirty) store_xi(a.env.xi, i, p);
        a.env.elapsed[i] = el;
        if (kLog) args.log.count[i] = (int32_t)log_count;
        if (a.env.episode && episodes) a.env.episode[i] += episodes;      // one started per episode that ended
    }
    rollout_publish(a.stats, a.violations, episodes, sum_len, sum_len, sum_r2, min_r, max_r, viol);
}

}  // namespace renv
