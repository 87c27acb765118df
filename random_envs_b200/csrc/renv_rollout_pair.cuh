// Fused K-step rollout, fp32, TWO envs per thread on Blackwell's packed FP32 pipe (FFMA2 / FMUL2:
// PTX fma.rn.f32x2 / mul.rn.f32x2, new in sm_100).
//
// Why: the one-env-per-thread rollout is bound by instruction ISSUE (ncu: issue-active 94 %, FMA pipe 60 %): ~45
// issue slots per env-step of which ~26 are FFMA/FMUL.  An FFMA2 does the same arithmetic for two envs in one
// issue slot (measured on B200: 3-register FFMA 49 TFLOP/s, FFMA2 64 TFLOP/s at 0.44x the issue slots), so a
// thread that owns an env PAIR spends 26 packed + ~14 scalar (compare / select / MUFU.RCP) slots per two env-steps.
// Every packed lane rounds exactly like the scalar FFMA/FMUL of renv_cartpole.cuh (same operation sequence; the
// negations of the scalar code are folded into pre-negated operands, which is exact), so the result is
// bit-identical to K launches of the single-step kernel -- tests/test_gpu_vecenv.py compares them with ==.
//
// Control flow without per-step bookkeeping: a thread counts its packed steps in ONE counter c.  Slot k (k = 0, 1)
// is described by B_k (env-steps done = B_k + c), E_k (elapsed = E_k + c) and L_k = the value of c at which it
// either hits the TimeLimit or has done its K steps; the hot loop tests `terminated_k || c >= L_k` and nothing
// else.  An inactive slot (parked for a deferred reset, finished, or beyond n) holds NaN state -- NaN never
// satisfies |x| > 2.4 -- and L_k = INT_MAX, so it needs no mask.  Resets are deferred and executed once per warp
// for several parked slots (see cartpole_rollout_kernel); a slot that finishes its K steps stores its env at once.
#pragma once
#include "renv_kernels.cuh"
#include "renv_pack.cuh"

namespace renv {

constexpr int kPairResetBatch = 16;      // parked slots (of 64) per warp that trigger a reset pass
constexpr int kPairCtas = 3;             // resident CTAs per SM (register cap)
constexpr int kPairSlots = 2;            // envs per thread: one packed pair
constexpr int kInactive = 0x7fffffff;

// Per-slot operands of the packed step, as scalars (the hot loop packs slot 0 / slot 1 into register pairs).
struct PairSlot {
    float x, xd, th, thd;                       // state
    float ng, fot, pmlot, l43, nlpm;            // -gravity, F/M, pml/M, l*4/3, -(l*m_p/M)   (Derived<float>)
    int B, E, L, parked;                        // see the header comment; parked = env-steps done when parked, -1 = not;
                                                // an inactive slot's E is the counter itself (see on_event)
    uint32_t log_count;                         // logged kernel only: episode-log records of the env (stored at exit)
};

__device__ __forceinline__ void slot_params(PairSlot &q, const Xi<float> &p)
{
    const Derived<float> d = derive(p);
    q.ng = -p.gravity; q.fot = d.force_over_total; q.pmlot = d.pml_over_total;
    q.l43 = d.len_four_thirds; q.nlpm = -d.len_pm_over_total;
}

// Loop-invariant packed operands of the step (policy weights from the kernel parameters, polynomial coefficients).
struct PairConsts {
    u64 W0, W1, W2, W3, WB, C120, CM6, CM720, C24, CMH, ONE, TAU, NTAU;
};

// One env-step for the env pair (s0, s1): policy_action<float> + sincos_small<true> + dynamics<float>, every operation
// the packed twin of the scalar one in renv_cartpole.cuh.  NNUM = -num and NTHACC = -theta_acc (exact: rounding is
// sign-symmetric), so no negation instructions are needed.
template <bool kEuler>
__device__ __forceinline__ void pair_step(PairSlot &s0, PairSlot &s1, const PairConsts &k)
{
    u64 X = pk(s0.x, s1.x), XD = pk(s0.xd, s1.xd), TH = pk(s0.th, s1.th), THD = pk(s0.thd, s1.thd);
    const u64 NG = pk(s0.ng, s1.ng), PMLOT = pk(s0.pmlot, s1.pmlot), L43 = pk(s0.l43, s1.l43), NLPM = pk(s0.nlpm, s1.nlpm);
    u64 acc = fma2(k.W0, X, k.WB);
    acc = fma2(k.W1, XD, acc);
    acc = fma2(k.W2, TH, acc);
    acc = fma2(k.W3, THD, acc);
    float acc0, acc1;
    unpk(acc, acc0, acc1);
    const u64 PUSH = pk(acc0 > 0.0f ? s0.fot : -s0.fot, acc1 > 0.0f ? s1.fot : -s1.fot);
    const u64 X2 = mul2(TH, TH);
    const u64 PS = fma2(X2, k.C120, k.CM6);
    const u64 SN = fma2(mul2(TH, X2), PS, TH);
    u64 PC = fma2(X2, k.CM720, k.C24);
    PC = fma2(X2, PC, k.CMH);
    const u64 CS = fma2(X2, PC, k.ONE);
    const u64 TEMP = fma2(mul2(mul2(THD, THD), SN), PMLOT, PUSH);
    const u64 NNUM = fma2(NG, SN, mul2(CS, TEMP));
    const u64 DEN = fma2(NLPM, mul2(CS, CS), L43);
    float den0, den1;
    unpk(DEN, den0, den1);
    const u64 NTHACC = mul2(NNUM, pk(rcp_approx(den0), rcp_approx(den1)));
    const u64 XACC = fma2(mul2(PMLOT, CS), NTHACC, TEMP);
    if (kEuler) {
        X = fma2(k.TAU, XD, X);
        XD = fma2(k.TAU, XACC, XD);
        TH = fma2(k.TAU, THD, TH);
        THD = fma2(k.NTAU, NTHACC, THD);
    } else {
        XD = fma2(k.TAU, XACC, XD);
        X = fma2(k.TAU, XD, X);
        THD = fma2(k.NTAU, NTHACC, THD);
        TH = fma2(k.TAU, THD, TH);
    }
    unpk(X, s0.x, s1.x); unpk(XD, s0.xd, s1.xd); unpk(TH, s0.th, s1.th); unpk(THD, s0.thd, s1.thd);
}

// kLog: on_event stores an ended episode's terminal state and length like a finished env's (one more use of a store
// the hot loop already has), and reset_slot -- in the warp's reset pass, outside the loop -- reads them back with the
// env's xi row (current in HBM: every reset stores it) and writes the episode-log record before the resample.
template <bool kEuler, bool kLog>
__device__ __forceinline__ void rollout_pair_body(const RolloutArgs<float> &a, const LogPtrs<float> &log)
{
    constexpr int S = kPairSlots;
    const int64_t i0 = S * ((int64_t)blockIdx.x * blockDim.x + threadIdx.x);
    const int64_t ld = a.env.ld, n = a.env.n;
    const int K = a.K;
    const int32_t limit = a.max_steps > 0 ? a.max_steps : 0x7fffffff;
    const float nan = __int_as_float(0x7fc00000);

    unsigned long long sum_r2 = 0;
    unsigned sum_r = 0, episodes = 0, viol = 0;
    float min_r = __int_as_float(0x7f800000), max_r = __int_as_float(0xff800000);
    int c = 0;                                   // packed steps executed by this thread
    PairSlot q[S];

    auto deactivate = [&](PairSlot &s) { s.x = nan; s.xd = nan; s.th = nan; s.thd = nan; s.L = kInactive; };
    auto activate = [&](PairSlot &s, int steps_done, int elapsed) {
        s.B = steps_done - c; s.E = elapsed - c;
        const long long lk = min((long long)K - s.B, (long long)limit - s.E);
        s.L = (int)min(lk, (long long)(kInactive - 1));
    };
    auto store_state = [&](const PairSlot &s, int64_t i) {
        a.env.state[i] = s.x; a.env.state[ld + i] = s.xd; a.env.state[2 * ld + i] = s.th; a.env.state[3 * ld + i] = s.thd;
    };
    // slot reached `terminated || c >= L`: the episode ended (-> statistics, park for the deferred reset) or the
    // env has done its K steps in a still-running episode (-> store its state, slot goes inactive).  Either way E
    // takes the counter's value: the ended episode's length (the reset pass logs it) or the env's final count, which
    // the kernel stores once at exit -- the counter is read at entry and written at exit, never in the loop
    auto on_event = [&](PairSlot &s, int64_t i, bool terminated) {
        const int steps_done = s.B + c, el = s.E + c;
        if (terminated || el >= limit) {
            const float ret = (float)el;
            episodes += 1; sum_r += (unsigned)el; sum_r2 += (unsigned long long)el * (unsigned)el;   // reward is 1.0/step
            min_r = fminf(min_r, ret); max_r = fmaxf(max_r, ret);
            s.parked = steps_done;
            if (kLog) store_state(s, i);
        } else {
            store_state(s, i);
        }
        s.E = el;
        deactivate(s);
    };
    // RandomCartPoleEnv.reset (+ set_random_task) at the clock tick of the step that ended the episode
    auto reset_slot = [&](PairSlot &s, int64_t i) {
        const uint64_t id = a.env.env_id0 + (uint64_t)i;
        const uint64_t tick = a.tick + (uint64_t)(s.parked - 1);
        if (kLog) {
            const State<float> fs = { a.env.state[i], a.env.state[ld + i], a.env.state[2 * ld + i], a.env.state[3 * ld + i] };
            const int32_t len = s.E;
            log_episode(log, ld, i, s.log_count, load_xi(a.env.xi, i), fs, len, !beyond_thresholds(fs) && len >= limit, tick);
            s.log_count += 1u;
        }
        if (a.dr.dr_type != kDrNone) {
            Xi<float> p = { 0.0f, 0.0f, 0.0f, 0.0f };
            viol += sample_xi(p, a.dr, a.env.seed, id, tick);
            store_xi(a.env.xi, i, p);
            slot_params(s, p);
        }
        State<float> st;
        init_state(st, a.env.seed, id, tick);
        s.x = st.x; s.xd = st.x_dot; s.th = st.theta; s.thd = st.theta_dot;
        if (a.env.episode) atomicAdd(a.env.episode + i, 1u);
        const int steps_done = s.parked;
        s.parked = -1;
        if (steps_done >= K) { store_state(s, i); s.E = 0; deactivate(s); }   // the episode ended on the launch's last step
        else activate(s, steps_done, 0);
    };

    // ---- load + step 0 (scalar: an injected state may have any angle; from step 1 on |theta| <= 0.2095) -------
    const Policy<float> policy = { a.policy.w0, a.policy.w1, a.policy.w2, a.policy.w3, a.policy.b };
    bool term0[S];
#pragma unroll
    for (int k = 0; k < S; ++k) {
        PairSlot &s = q[k];
        const int64_t i = i0 + k;
        term0[k] = false;
        s.parked = -1; s.B = 0; s.E = 0;
        s.ng = -1.0f; s.fot = 1.0f; s.pmlot = 1.0f; s.l43 = 1.0f; s.nlpm = -0.5f;
        if (i < n) {
            State<float> st = { a.env.state[i], a.env.state[ld + i], a.env.state[2 * ld + i], a.env.state[3 * ld + i] };
            const Xi<float> p = load_xi(a.env.xi, i);
            slot_params(s, p);
            term0[k] = dynamics<false>(st, p, derive(p), policy_action(policy, st), kEuler);
            s.x = st.x; s.xd = st.x_dot; s.th = st.theta; s.thd = st.theta_dot;
            activate(s, 0, load_elapsed(a.env, i));
            if (kLog) s.log_count = (uint32_t)log.count[i];     // in a register: no DRAM round trip in the reset pass
        } else {
            deactivate(s);
        }
    }
    c = 1;
#pragma unroll
    for (int k = 0; k < S; ++k)
        if (i0 + k < n && (term0[k] || c >= q[k].L)) on_event(q[k], i0 + k, term0[k]);

    const PairConsts kc = { splat(policy.w0), splat(policy.w1), splat(policy.w2), splat(policy.w3), splat(policy.b),
                            splat(1.0f / 120.0f), splat(-1.0f / 6.0f), splat(-1.0f / 720.0f), splat(1.0f / 24.0f),
                            splat(-0.5f), splat(1.0f), splat((float)kTau), splat(-(float)kTau) };
    const float xthr = (float)kXThreshold, ththr = (float)kThetaThreshold;

    for (;;) {
#pragma unroll
        for (int u = 0; u < kStepsPerCheck; ++u) {
            pair_step<kEuler>(q[0], q[1], kc);
            c += 1;
            bool term[S], any = false;
#pragma unroll
            for (int k = 0; k < S; ++k) {
                term[k] = fabsf(q[k].x) > xthr || fabsf(q[k].th) > ththr;
                any = any || term[k] || c >= q[k].L;
            }
            if (any) {
#pragma unroll
                for (int k = 0; k < S; ++k)
                    if (term[k] || c >= q[k].L) on_event(q[k], i0 + k, term[k]);
            }
        }
        int nparked = 0;
        bool active = false, parked = false;
#pragma unroll
        for (int k = 0; k < S; ++k) {
            nparked += __popc(__ballot_sync(0xffffffffu, q[k].parked >= 0));
            active = active || q[k].L != kInactive;
            parked = parked || q[k].parked >= 0;
        }
        const unsigned running = __ballot_sync(0xffffffffu, active);
        if (nparked != 0 && (nparked >= kPairResetBatch || running == 0u)) {
            if (parked) {
#pragma unroll
                for (int k = 0; k < S; ++k)
                    if (q[k].parked >= 0) reset_slot(q[k], i0 + k);
            }
            continue;                       // revived slots may still have steps to do
        }
        if (running == 0u) break;
    }
#pragma unroll
    for (int k = 0; k < S; ++k) {        // every slot of an env has finished: E is its counter
        if (i0 + k < n) {
            store_elapsed(a.env, i0 + k, q[k].E);
            if (kLog) log.count[i0 + k] = (int32_t)q[k].log_count;
        }
    }
    rollout_publish(a.stats, a.violations, episodes, sum_r, sum_r, sum_r2, min_r, max_r, viol);
}

template <bool kEuler>
__global__ void __launch_bounds__(kRolloutThreads, kPairCtas)
cartpole_rollout_pair_kernel(const __grid_constant__ RolloutArgs<float> a)
{
    rollout_pair_body<kEuler, false>(a, LogPtrs<float>{});
}

template <bool kEuler>
__global__ void __launch_bounds__(kRolloutThreads, kPairCtas)
cartpole_rollout_pair_logged_kernel(const __grid_constant__ LoggedRolloutArgs<float> a)
{
    rollout_pair_body<kEuler, true>(a.roll, a.log);
}

}  // namespace renv
