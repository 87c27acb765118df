// Body of cartpole_rollout_mlp_kernel, cartpole_collect_mlp_kernel, cartpole_population_mlp_kernel,
// cartpole_grid_mlp_kernel, cartpole_scen_rollout_mlp_kernel, cartpole_scen_collect_mlp_kernel,
// cartpole_mix_rollout_mlp_kernel and cartpole_mix_collect_mlp_kernel (renv_mlp_policy.cuh), included textually into
// each of these __global__ functions so that the rollout compiles to exactly the code it had before the other kernels
// existed (an inlined device function would not guarantee that: DESIGN.md section 4.8).  The including function defines
//     kAct, kEuler, kLog, kCollect, kPop, kGrid, kScen, kMix   (template parameters or constexpr)
//     args     the launch arguments: .roll (RolloutArgs<float>), .params, .log (read only when kLog)
//     traj     const MlpTrajPtrs &: the per-step record (read only when kCollect)
//     sample   bool: sample the action from softmax(l0, l1) instead of taking the argmax (read only when kCollect)
//     kPop, pop   cartpole_population_mlp_kernel (PopulationPtrs, read only when kPop): CTA b serves envs
//                 (b % pop.ctas) * kMlpThreads + threadIdx.x of member b / pop.ctas, whose parameters are row
//                 b / pop.ctas of pop.policies, from a fresh episode started in registers at tick a.tick - 1; it stores
//                 nothing into the env and publishes into the member's stats row
//     kGrid, grid cartpole_grid_mlp_kernel (with kPop; GridPtrs, read only when kGrid): pop.ctas = ceil(C n / 128), and
//                 the CTA's index i runs over the member's flat (scenario, env) range, i < grid.span = C n: lane i serves
//                 env j = i % n under scenario c = i / n, whose row replaces a.dr / the env's table, and publishes
//                 into cell p C + c's stats row by population_publish (a CTA may span several cells)
//     kScen, env_scen  the per-env scenario kernels (EnvScenPtrs, read only when kScen): lane i reads env i's scenario
//                 index once here and its row (global memory) at resets only; the row replaces a.dr, a fixed-task row's
//                 task replaces the env's xi at each reset, and statistics go to the scenario's row (scenario_publish)
//     kMix, mix   the mixture kernels (MixPtrs, read only when kMix): each reset draws the lane's row (mixture_draw),
//                 which then acts as a kScen row; the running sums belong to the row of the current episode and are
//                 flushed when a reset draws another row (mixture_stats_add); of_env is stored at the end
// No include guard: included once per kernel.
    __shared__ MlpSmem sm;
    const uint32_t member = kPop ? blockIdx.x / pop.ctas : 0u;
    mlp_load_params(sm, kPop ? pop.policies + (size_t)member * kMlpParamFloats : args.params);
    const RolloutArgs<float> &a = args.roll;
    const int64_t i = (int64_t)(kPop ? blockIdx.x - member * pop.ctas : blockIdx.x) * blockDim.x + threadIdx.x;
    const int64_t ld = a.env.ld;
    const bool live = i < (kGrid ? (int64_t)grid.span : a.env.n);
    // kGrid: lanes past C n shadow the last scenario (C n < 2^31: 32-bit division)
    const uint32_t grid_scenario_of = kGrid ? (uint32_t)(live ? i : grid.span - 1) / (uint32_t)a.env.n : 0u;
    const int64_t il = kGrid ? (live ? i - (int64_t)grid_scenario_of * a.env.n : 0) : live ? i : 0;
    const uint32_t scenario = kScen ? env_scenario(env_scen, il) : grid_scenario_of;
    const uint64_t id = a.env.env_id0 + (uint64_t)il;
    const DrCfg4<float> &dr = kGrid ? grid_scenario<float>(grid, scenario)
                            : kScen ? scenario_row<float>(env_scen.rows, scenario) : a.dr;
    uint32_t mix_row = kMix ? min((uint32_t)mix.of_env[il], mix.C) : 0u;    // kMix: the row of the running episode
    unsigned mix_ended = 0;                 // kMix: episodes ended (the running sums restart at each flush)
    if (kMix) mixture_stats_begin(mix.C);

    State<float> s;
    Xi<float> p;
    unsigned fresh_viol = 0;
    if (kPop) {         // renv_cartpole_reset_f32 at tick a.tick - 1, in registers (lanes past n shadow env 0)
        init_state(s, a.env.seed, id, a.tick - 1);
        if (draws_xi<kGrid>(dr.dr_type)) {
            p = Xi<float>{ 0.0f, 0.0f, 0.0f, 0.0f };
            const unsigned v = sample_xi(p, dr, a.env.seed, id, a.tick - 1);
            fresh_viol = live ? v : 0u;
        } else if (kGrid) {     // a fixed-task scenario: its task, kept across resets
            p = Xi<float>{ dr.a[0], dr.a[1], dr.a[2], dr.a[3] };
        } else {
            p = load_xi(a.env.xi, il);
        }
    } else {
        s = live ? State<float>{ a.env.state[i], a.env.state[ld + i], a.env.state[2 * ld + i], a.env.state[3 * ld + i] }
                 : State<float>{ 0.0f, 0.0f, 0.0f, 0.0f };      // lanes past n feed zero rows
        p = load_xi(a.env.xi, il);
    }
    Derived<float> d = derive(p);
    int32_t el = kPop ? 0 : load_elapsed(a.env, il);
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
                    if (kMix) mix_ended += 1u;
                    const uint32_t c = kMix ? mixture_draw(mix, a.env.seed, id, tick) : 0u;
                    const DrCfg4<float> &rdr = kMix ? scenario_row<float>(mix.rows, c) : dr;
                    if (draws_xi<kGrid || kScen || kMix>(rdr.dr_type)) {   // reset_env: set_random_task, then reset
                        p = Xi<float>{ 0.0f, 0.0f, 0.0f, 0.0f };
                        viol += sample_xi(p, rdr, a.env.seed, id, tick);
                        d = derive(p);
                        xi_dirty = true;
                    } else if (kScen || kMix) {                            // a fixed-task row: its task
                        p = Xi<float>{ rdr.a[0], rdr.a[1], rdr.a[2], rdr.a[3] };
                        d = derive(p);
                        xi_dirty = true;
                    }
                    init_state(s, a.env.seed, id, tick);
                    if (kMix && c != mix_row) {     // the ended episode was the last of row mix_row in this run
                        mixture_stats_add(a.stats, mix.C, mix_row, episodes, sum_len, sum_len, sum_r2, min_r, max_r);
                        episodes = 0; sum_len = 0; sum_r2 = 0;
                        min_r = __int_as_float(0x7f800000); max_r = __int_as_float(0xff800000);
                        mix_row = c;
                    }
                }
            }
            __syncwarp();
        }
    }

    if (live && !kPop) {
        a.env.state[i] = s.x; a.env.state[ld + i] = s.x_dot; a.env.state[2 * ld + i] = s.theta; a.env.state[3 * ld + i] = s.theta_dot;
        if (xi_dirty) store_xi(a.env.xi, i, p);
        store_elapsed(a.env, i, el);
        if (kLog) args.log.count[i] = (int32_t)log_count;
        if (kMix) mix.of_env[i] = (uint16_t)mix_row;
        if (kMix) {
            if (a.env.episode && mix_ended) a.env.episode[i] += mix_ended;
        } else if (a.env.episode && episodes) a.env.episode[i] += episodes;      // one started per episode that ended
    }
    if (kGrid) {
        const int64_t cell = (int64_t)member * grid.C + scenario;
        population_publish(a.stats + 6 * cell, cell, a.violations, episodes, sum_len, sum_len, sum_r2, min_r, max_r, viol);
    } else if (kMix) {
        mixture_stats_add(a.stats, mix.C, mix_row, episodes, sum_len, sum_len, sum_r2, min_r, max_r);
        mixture_stats_end(a.stats, mix.C, a.violations, viol);
    } else if (kScen) {
        scenario_publish(a.stats, env_scen.C, scenario, a.violations, episodes, sum_len, sum_len, sum_r2, min_r, max_r, viol);
    } else {
        rollout_publish(kPop ? a.stats + 6 * member : a.stats, a.violations, episodes, sum_len, sum_len, sum_r2, min_r, max_r, viol);
    }
