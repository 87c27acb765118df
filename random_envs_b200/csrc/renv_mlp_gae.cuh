// Advantage estimation under an MLP critic (include/renv.h renv_cartpole_gae_mlp_f32): the values, GAE advantages and
// returns of a trajectory cartpole_collect_mlp_kernel has just written, in one launch.
//
// The critic is a packed 1-output net (renv_mlp_policy with l0 = 0): V(s) = l1 of mlp_logits(), the same function and
// therefore the same bits as every other MLP kernel (policy_actions' logits column 1 for state s).  Per env, from the
// last step backwards, with v_K = V(s_K) (the env's state after the collect), A_K = 0 and gl = gamma * lambda:
//
//     v_k   = V(obs[k])
//     nv_k  = done[k] ? (truncated[k] ? V(final_obs[k]) : 0) : v_{k+1}
//     delta = (1 + gamma nv_k) - v_k
//     A_k   = done[k] ? delta : delta + gl A_{k+1}
//     R_k   = A_k + v_k
//
// Every operation is an explicit round-to-nearest intrinsic, so nothing is contracted into an FMA and a float32 host
// replay of these lines reproduces advantages and returns bit for bit from the stored values.
//
// Launch as the MLP rollout: 128 threads per CTA, one env per lane, the critic staged once per CTA in shared memory and
// all lanes of a warp in lockstep over the K steps (mma.sync is warp-collective).  Lanes past n feed a zero state; a
// warp entirely past n returns after the staging barrier.  V(final_obs) is a second mlp_logits pass, run only on the
// steps where some lane of the warp was truncated (about 6 % of warp-steps with 500-step episodes).
#pragma once
#include "renv_mlp_policy.cuh"

namespace renv {

struct MlpGaeArgs {
    const float *state; int64_t n, ld;    // the env's SoA state: s_K
    const float *params;                  // the packed critic
    const float *obs, *final_obs;         // (capacity, ld, 4) rows
    const uint8_t *done, *truncated;      // (capacity, ld)
    float *values, *advantages, *returns; // (capacity, ld)
    int K;
    float gamma, lambda;
};

// V(s) for this lane's env; warp-collective like mlp_logits.  The kernel inlines it three times (V(s_K), V(obs),
// V(final_obs)); the compiler barrier keeps the compiler from merging the copies' shared-memory loads of the weights
// into values kept live across the K loop (without it ptxas spills ~1.4 KB per thread).
template <int kAct> __device__ __forceinline__ float mlp_value(const MlpSmem &sm, const State<float> &s)
{
    asm volatile("" ::: "memory");
    float l0, l1;
    mlp_logits<kAct>(sm, s, l0, l1);
    return l1;
}

__device__ __forceinline__ State<float> load_row(const float *rows, int64_t r)
{
    const float4 v = *reinterpret_cast<const float4 *>(rows + 4 * r);
    return State<float>{ v.x, v.y, v.z, v.w };
}

template <int kAct>
__global__ void __launch_bounds__(kMlpThreads, kMlpRolloutCtas)
cartpole_gae_mlp_kernel(const __grid_constant__ MlpGaeArgs a)
{
    __shared__ MlpSmem sm;
    mlp_load_params(sm, a.params);
    const int64_t base = (int64_t)blockIdx.x * kMlpThreads;
    if (base + (threadIdx.x & ~31) >= a.n) return;              // the whole warp is past n (warp-uniform)
    const int64_t i = base + threadIdx.x, ld = a.ld;
    const bool live = i < a.n;
    const State<float> zero{ 0.0f, 0.0f, 0.0f, 0.0f };
    const float gamma = a.gamma, gl = __fmul_rn(a.gamma, a.lambda);

    float v_next = mlp_value<kAct>(sm, live ? State<float>{ a.state[i], a.state[ld + i], a.state[2 * ld + i],
                                                            a.state[3 * ld + i] } : zero);     // V(s_K)
    float adv = 0.0f;                                                                          // A_K
    for (int k = a.K - 1; k >= 0; --k) {
        const int64_t row = (int64_t)k * ld + i;
        const State<float> s = live ? load_row(a.obs, row) : zero;
        const bool done = live && a.done[row] != 0;
        const bool trunc = done && a.truncated[row] != 0;
        const float v = mlp_value<kAct>(sm, s);
        float nv = done ? 0.0f : v_next;
        if (__any_sync(0xffffffffu, trunc)) {                   // warp-uniform: the bootstrap of truncated episodes
            const float vf = mlp_value<kAct>(sm, trunc ? load_row(a.final_obs, row) : zero);
            if (trunc) nv = vf;
        }
        const float delta = __fsub_rn(__fadd_rn(1.0f, __fmul_rn(gamma, nv)), v);
        adv = done ? delta : __fadd_rn(delta, __fmul_rn(gl, adv));
        if (live) {
            a.values[row] = v;
            a.advantages[row] = adv;
            a.returns[row] = __fadd_rn(adv, v);
        }
        v_next = v;
    }
}

}  // namespace renv
