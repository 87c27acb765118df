// Body of cartpole_rollout_mlp_kernel, cartpole_collect_mlp_kernel and cartpole_population_mlp_kernel
// (renv_mlp_policy.cuh), included textually into each of these __global__ functions so that the rollout compiles to
// exactly the code it had before the other kernels existed (an inlined device function would not guarantee that:
// DESIGN.md section 4.8).  The including function defines
//     kAct, kEuler, kLog, kCollect, kPop   (template parameters or constexpr)
//     args     the launch arguments: .roll (RolloutArgs<float>), .params, .log (read only when kLog)
//     traj     const MlpTrajPtrs &: the per-step record (read only when kCollect)
//     sample   bool: sample the action from softmax(l0, l1) instead of taking the argmax (read only when kCollect)
//     kPop, pop   cartpole_population_mlp_kernel (PopulationPtrs, read only when kPop): CTA b serves envs
//                 (b % pop.ctas) * kMlpThreads + threadIdx.x of member b / pop.ctas, whose parameters are row
//                 b / pop.ctas of pop.policies, from a fresh episode started in registers at tick a.tick - 1; it stores
//                 nothing into the env and publishes into the member's stats row
// No include guard: included once per kernel.
    __shared__ MlpSmem sm;
    const uint32_t member = kPop ? blockIdx.x / pop.ctas : 0u;
    mlp_load_params(sm, kPop ? pop.policies + (size_t)member * kMlpParamFloats : args.params);
    const RolloutArgs<float> &a = args.roll;
    const int64_t i = (int64_t)(kPop ? blockIdx.x - member * pop.ctas : blockIdx.x) * blockDim.x + threadIdx.x;
    const int64_t ld = a.env.ld;
    const bool live = i < a.env.n;
    const int64_t il = live ? i : 0;
    const uint64_t id = a.env.env_id0 + (uint64_t)il;

    State<float> s;
    Xi<float> p;
    unsigned fresh_viol = 0;
    if (kPop) {         // renv_cartpole_reset_f32 at tick a.tick - 1, in registers (lanes past n shadow env 0)
        init_state(s, a.env.seed, id, a.tick - 1);
        if (a.dr.dr_type != kDrNone) {
            p = Xi<float>{ 0.0f, 0.0f, 0.0f, 0.0f };
            const unsigned v = sample_xi(p, a.dr, a.env.seed, id, a.tick - 1);
            fresh_viol = live ? v : 0u;
        } else {
            p = load_xi(a.env.xi, il);
        }
    } else {
        s = live ? State<float>{ a.env.state[i], a.env.state[ld + i], a.env.state[2 * ld + i], a.env.state[3 * ld + i] }
                 : State<float>{ 0.0f, 0.0f, 0.0f, 0.0f };      // lanes past n feed zero rows
        p = load_xi(a.env.xi, il);
    }
    Derived<float> d = derive(p);
    int32_t el = kPop ? 0 : a.env.elapsed[il];
    uint32_t log_count = kLog ? (uint32_t)args.log.count[il] : 0u;
    unsigned episodes = 0, sum_len = 0, viol = fresh_viol;   // return == length (:207-212): sum_len is also sum R
    unsigned long long sum_r2 = 0;
    float min_r = __int_as_float(0x7f800000), max_r = __int_as_float(0xff800000);
    bool xi_dirty = false;

    if (__any_sync(0xffffffffu, live)) {                        // warp-uniform: a warp entirely past n only publishes
        for (int k = 0; k < a.K; ++k) {
            float l0, l1;
            mlp_logits<kAct>(sm, s, l0, l1);
            if (live) {
                const int64_t row = (int64_t)k * ld + i;                   // trajectory row of this step (kCollect)
                float logp = 0.0f;
                const int action = kCollect ? mlp_pick(l0, l1, sample, a.env.seed, id, a.tick + (uint64_t)k, logp)
                                            : mlp_action(l0, l1);
                if (kCollect) {                                            // the observation the action was chosen from
                    store_xi(traj.obs, row, Xi<float>{ s.x, s.x_dot, s.theta, s.theta_dot });
                    traj.action[row] = (uint8_t)action;
                    if (traj.logp) traj.logp[row] = logp;
                }
                // step 0 may start from an injected state at any angle; from step 1 on |theta| <= 0.2095 holds at
                // every step start (an env beyond the threshold was just reset): the same bits without the range check.
                // A population member starts from a reset state: no check at step 0 either.
                const bool terminated = k == 0 && !kPop ? dynamics<false>(s, p, d, action, kEuler)
                                                        : dynamics<true>(s, p, d, action, kEuler);
                el += 1;                                                   // TimeLimit.step
                if (kCollect) {
                    const bool truncated = !terminated && a.max_steps > 0 && el >= a.max_steps;
                    traj.done[row] = (uint8_t)(terminated || truncated);
                    if (traj.truncated) traj.truncated[row] = (uint8_t)truncated;
                }
                if (terminated || (a.max_steps > 0 && el >= a.max_steps)) {
                    const uint64_t tick = a.tick + (uint64_t)k;
                    const float ret = (float)el;
                    episodes += 1; sum_len += (unsigned)el;
                    sum_r2 += (unsigned long long)el * (unsigned)el;
                    min_r = fminf(min_r, ret); max_r = fmaxf(max_r, ret);
                    if (kCollect && traj.final_obs)                        // the terminal observation auto-reset replaces
                        store_xi(traj.final_obs, row, Xi<float>{ s.x, s.x_dot, s.theta, s.theta_dot });
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

    if (live && !kPop) {
        a.env.state[i] = s.x; a.env.state[ld + i] = s.x_dot; a.env.state[2 * ld + i] = s.theta; a.env.state[3 * ld + i] = s.theta_dot;
        if (xi_dirty) store_xi(a.env.xi, i, p);
        a.env.elapsed[i] = el;
        if (kLog) args.log.count[i] = (int32_t)log_count;
        if (a.env.episode && episodes) a.env.episode[i] += episodes;      // one started per episode that ended
    }
    rollout_publish(kPop ? a.stats + 6 * member : a.stats, a.violations, episodes, sum_len, sum_len, sum_r2, min_r, max_r, viol);
