// Body of cartpole_rollout_kernel, cartpole_rollout_logged_kernel and cartpole_population_linear_kernel
// (renv_kernels.cuh), included textually into each of these __global__ functions for the reason given in
// renv_step_body.cuh.  The including function defines
//     T, kEuler, kNoisy, kRandom, kLog, kPop   (template parameters or constexpr)
//     a    const RolloutArgs<T> &  the launch arguments
//     log  const LogPtrs<T> &      the episode log (read only when kLog): an ended episode's record is written in the
//                                  warp's reset pass, before rollout_reset overwrites t.s / t.p / t.el
//     kPop (constexpr), pop (PopulationPtrs, read only when kPop): cartpole_population_linear_kernel.  Thread i serves
//          env j = i % n of member i / n (i < pop.total = P n), from a fresh episode started in registers at tick
//          a.tick - 1, under member's policy row; it stores nothing into the env and publishes into member's stats row.
// No include guard: included once per kernel.
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t ld = a.env.ld;
    const bool live = i < (kPop ? pop.total : a.env.n);
    // dead lanes of the last warp shadow the last member's env 0 with zero steps to do (P n < 2^31: 32-bit division)
    const int64_t member = kPop ? (int64_t)((uint32_t)(live ? i : pop.total - 1) / (uint32_t)a.env.n) : 0;
    const int64_t il = kPop ? (live ? i - member * a.env.n : 0) : live ? i : 0;

    // per-thread episode statistics (return == length here: reward is 1.0 on every step, :207-212)
    RolloutThread<T> t;
    t.sum_r = 0; t.sum_r2 = 0;
    t.min_r = __int_as_float(0x7f800000); t.max_r = __int_as_float(0xff800000);
    t.episodes = 0; t.sum_len = 0; t.viol = 0;
    if (kPop) {         // renv_cartpole_reset_f32 at tick a.tick - 1, in registers
        init_state(t.s, a.env.seed, a.env.env_id0 + (uint64_t)il, a.tick - 1);
        if (a.dr.dr_type != kDrNone) {
            t.p = Xi<T>{ T(0), T(0), T(0), T(0) };
            const unsigned v = sample_xi(t.p, a.dr, a.env.seed, a.env.env_id0 + (uint64_t)il, a.tick - 1);
            t.viol = live ? v : 0u;
        } else {
            t.p = load_xi(a.env.xi, il);
        }
    } else {
        t.s = State<T>{ a.env.state[il], a.env.state[ld + il], a.env.state[2 * ld + il], a.env.state[3 * ld + il] };
        t.p = load_xi(a.env.xi, il);
    }
    t.d = derive(t.p);
    t.el = kPop ? 0 : a.env.elapsed[il];
    t.new_episodes = 0; t.xi_dirty = false; t.parked = -1;
    t.obs_loaded = kNoisy; t.after_reset = 0u;
    t.act.group = (uint32_t)a.tick >> 7; t.act.r = make_uint4(0, 0, 0, 0); t.refresh = false;
    if (kRandom) t.act.r = draw_block(a.env.seed, a.env.env_id0 + (uint64_t)il, (uint64_t)t.act.group, kAction, 0);
    if (kNoisy) t.obs0 = State<T>{ a.env.obs[il], a.env.obs[ld + il], a.env.obs[2 * ld + il], a.env.obs[3 * ld + il] };
    else t.obs0 = t.s;
    const uint64_t id = a.env.env_id0 + (uint64_t)il;
    const int32_t limit = a.max_steps > 0 ? a.max_steps : 0x7fffffff;
    uint32_t log_count = kLog ? (uint32_t)log.count[il] : 0u;    // episode-log records of this env
    t.remaining = live ? a.K : 0;
    const float *const row = pop.policies + 5 * member;
    const Policy<T> policy = kPop ? Policy<T>{ pin(row[0]), pin(row[1]), pin(row[2]), pin(row[3]), pin(row[4]) }
                                  : Policy<T>{ pin(a.policy.w0), pin(a.policy.w1), pin(a.policy.w2), pin(a.policy.w3), pin(a.policy.b) };

    // Step 0 may start from a user-injected state with any angle; from step 1 on |theta| <= 0.2095 holds at
    // every step start (an env beyond the threshold was just reset), so the sin/cos range check is dropped.  A
    // population member starts from a reset state (|theta| <= 0.05): no check at step 0 either.
    if (t.remaining > 0) rollout_step<T, kEuler, kPop, kNoisy, kRandom>(t, a, policy, limit, id);
    for (;;) {
        if (sizeof(T) == 4 && !kNoisy && !kRandom) {
#pragma unroll
            for (int u = 0; u < kStepsPerCheck; ++u)
                if (t.remaining > 0) rollout_step<T, kEuler, true, kNoisy, kRandom>(t, a, policy, limit, id);
        } else if (kRandom && sizeof(T) == 4) {
#pragma unroll kRandomUnroll
            for (int u = 0; u < kRandomStepsPerCheck; ++u)
                if (t.remaining > 0) rollout_step<T, kEuler, true, kNoisy, kRandom>(t, a, policy, limit, id);
        } else {            // the fp64 / noisy step is ~10x the code of the fp32 one: keep the loop body inside the i-cache
#pragma unroll kUnrollF64
            for (int u = 0; u < kStepsPerCheck; ++u)
                if (t.remaining > 0) rollout_step<T, kEuler, true, kNoisy, kRandom>(t, a, policy, limit, id);
        }
        const unsigned parked = __ballot_sync(0xffffffffu, t.parked >= 0);
        const unsigned running = __ballot_sync(0xffffffffu, t.remaining > 0);
        if (parked != 0u && (__popc(parked) >= (kRandom && sizeof(T) == 4 ? kRandomResetBatch : kResetBatch) || running == 0u)) {
            if (t.parked >= 0) {
                if (kLog && !(kRandom && t.refresh)) {      // t.s / t.p / t.el are still the ended episode's
                    log_episode(log, ld, il, log_count, t.p, t.s, t.el, !beyond_thresholds(t.s) && t.el >= limit,
                                a.tick + (uint64_t)(a.K - t.parked - 1));
                    log_count += 1u;
                }
                rollout_reset<T, kRandom>(t, a, id);
            }
            continue;                       // revived lanes may still have steps to do
        }
        if (running == 0u) break;           // nobody parked, nobody running
    }

    if (live && !kPop) {
        a.env.state[i] = t.s.x; a.env.state[ld + i] = t.s.x_dot; a.env.state[2 * ld + i] = t.s.theta;
        a.env.state[3 * ld + i] = t.s.theta_dot;
        if (t.xi_dirty) store_xi(a.env.xi, i, t.p);
        a.env.elapsed[i] = t.el;
        if (kLog) log.count[i] = (int32_t)log_count;
        if (a.env.episode && t.new_episodes) a.env.episode[i] += t.new_episodes;
        if (kNoisy) {       // leave the obs buffer as K calls of step() would: the observation of the last step / reset
            T ov[4];
            add_obs_noise(t.s, a.env.noise_std, a.env.seed, id, a.tick + (uint64_t)(a.K - 1), t.after_reset, ov);
            a.env.obs[i] = ov[0]; a.env.obs[ld + i] = ov[1]; a.env.obs[2 * ld + i] = ov[2]; a.env.obs[3 * ld + i] = ov[3];
        }
    }
    if (kPop)
        population_publish(a.stats + 6 * member, member, a.violations, t.episodes, t.sum_len, t.sum_r, t.sum_r2, t.min_r,
                           t.max_r, t.viol);
    else
        rollout_publish(a.stats, a.violations, t.episodes, t.sum_len, t.sum_r, t.sum_r2, t.min_r, t.max_r, t.viol);
