// Body of cartpole_rollout_kernel and cartpole_rollout_logged_kernel (renv_kernels.cuh), included textually into both
// __global__ functions for the reason given in renv_step_body.cuh.  The including function defines
//     T, kEuler, kNoisy, kRandom, kLog         (template parameters or constexpr)
//     a    const RolloutArgs<T> &  the launch arguments
//     log  const LogPtrs<T> &      the episode log (read only when kLog): an ended episode's record is written in the
//                                  warp's reset pass, before rollout_reset overwrites t.s / t.p / t.el
// No include guard: included once per kernel.
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int64_t ld = a.env.ld;
    const bool live = i < a.env.n;
    const int64_t il = live ? i : 0;        // dead lanes of the last warp shadow env 0 with zero steps to do

    // per-thread episode statistics (return == length here: reward is 1.0 on every step, :207-212)
    RolloutThread<T> t;
    t.sum_r = 0; t.sum_r2 = 0;
    t.min_r = __int_as_float(0x7f800000); t.max_r = __int_as_float(0xff800000);
    t.episodes = 0; t.sum_len = 0; t.viol = 0;
    t.s = State<T>{ a.env.state[il], a.env.state[ld + il], a.env.state[2 * ld + il], a.env.state[3 * ld + il] };
    t.p = load_xi(a.env.xi, il);
    t.d = derive(t.p);
    t.el = a.env.elapsed[il];
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
    const Policy<T> policy = { pin(a.policy.w0), pin(a.policy.w1), pin(a.policy.w2), pin(a.policy.w3), pin(a.policy.b) };

    // Step 0 may start from a user-injected state with any angle; from step 1 on |theta| <= 0.2095 holds at
    // every step start (an env beyond the threshold was just reset), so the sin/cos range check is dropped.
    if (t.remaining > 0) rollout_step<T, kEuler, false, kNoisy, kRandom>(t, a, policy, limit, id);
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

    if (live) {
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
    rollout_publish(a.stats, a.violations, t.episodes, t.sum_len, t.sum_r, t.sum_r2, t.min_r, t.max_r, t.viol);
