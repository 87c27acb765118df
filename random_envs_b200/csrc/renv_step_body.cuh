// Body of cartpole_step_kernel, cartpole_step_logged_kernel, cartpole_scen_step_kernel and cartpole_mix_step_kernel
// (renv_kernels.cuh), included textually into each __global__ function rather than called as an inlined device
// function: an inlined body schedules the plain kernels' code differently, and the plain kernels must stay exactly what
// they were.  The including function defines
//     T, kAutoReset, kNoisy, kLean, kLog, kScen, kMix   (template parameters or constexpr; kLean is a per-launch
//                                                      constant in the logged kernel)
//     a    const StepArgs<T> &    the launch arguments
//     log  const LogPtrs<T> &     the episode log (read only when kLog)
//     env_scen  const EnvScenPtrs &  per-env scenarios (read only when kScen): the reset pass takes env i's row in
//                                    place of a.dr
//     mix  const MixPtrs &        a scenario mixture (read only when kMix): the reset pass draws env i's row, resets
//                                 from it and stores it in of_env
// No include guard: included once per kernel.
    using VT = VecTraits<T>;
    constexpr int V = VT::V;
    constexpr int kTile = kStepThreads * V;
    __shared__ unsigned s_count;
    __shared__ uint32_t s_ticket;                          // kScen, kMix: the ticket waits here across the reset pass
    __shared__ uint16_t s_list[kAutoReset ? kTile : 1];
    __shared__ int32_t s_len[kLog ? kTile : 1];          // length of the ended episode, negated when truncated
    const int64_t block0 = (int64_t)blockIdx.x * kTile;
    const int64_t i0 = block0 + (int64_t)threadIdx.x * V;
    const int64_t n = a.env.n, ld = a.env.ld;
    const bool live = i0 < n;
    const bool full = i0 + V <= n;
    const bool tracked = a.env.progress != nullptr;
    uint32_t ticket = 0;

    if (tracked) {
        if (threadIdx.x == 0) {
            uint32_t *const slot = a.env.progress + 2 * (size_t)blockIdx.x;
            ticket = atomicAdd(slot, 1u);
            uint32_t seen = ld_acquire_gpu(slot + 1);
            for (int spin = 0; seen != ticket && spin < kOrderSpins; ++spin) {     // rare: the predecessor is still on this tile
                __nanosleep(32);
                seen = ld_acquire_gpu(slot + 1);
            }
            if (seen != ticket && a.counters) atomicAdd(a.counters + kCounterOrderTimeout, 1ull);
            if (kScen || kMix) s_ticket = ticket;
            if (kAutoReset) s_count = 0;
        } else if (block0 + kTile <= n && threadIdx.x >= 32 && threadIdx.x < 39) {
            // while thread 0 waits for its L2 round trip the tile is pulled from HBM into L2 (never stale: L2 is the
            // point of coherence), so the loads below pay an L2 hit instead of a second DRAM latency
            const int q = threadIdx.x - 32;
            if (q < 4) prefetch_l2(a.env.state + q * ld + block0, kTile * sizeof(T));
            else if (q == 4) prefetch_l2(a.env.xi + 4 * block0, kTile * 4 * sizeof(T));
            else if (q == 5) { if (kLean) prefetch_l2(a.env.elapsed16 + block0, kTile * 2); else prefetch_l2(a.env.elapsed + block0, kTile * 4); }
            else prefetch_l2(a.action + block0, kTile);
        }
        __syncthreads();            // thread 0 holds the ticket and has seen the predecessor's release
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    } else {
        asm volatile("griddepcontrol.wait;" ::: "memory");
    }

    T s[4][V];
    Xi<T> p[V];
    int32_t el[V];
    uint8_t act[V];
    if (full) {     // all ten 128-bit requests go out before anything waits (incl. the barrier below)
#pragma unroll
        for (int c = 0; c < 4; ++c) vload<typename VT::Real>(s[c], a.env.state + c * ld + i0);
#pragma unroll
        for (int v = 0; v < V; ++v) p[v] = load_xi(a.env.xi, i0 + v);
        if (kLean) {
            uint16_t e16[V];
            vload<typename VT::Half>(e16, a.env.elapsed16 + i0);
#pragma unroll
            for (int v = 0; v < V; ++v) el[v] = e16[v];
        } else {
            vload<typename VT::Int>(el, a.env.elapsed + i0);
        }
        vload<typename VT::Byte>(act, a.action + i0);
    }
    if (kAutoReset && !tracked) {
        if (threadIdx.x == 0) s_count = 0;
        __syncthreads();            // overlaps the loads' latency
    }

    if (live) {
        if (!full) {
#pragma unroll
            for (int v = 0; v < V; ++v) {
                const bool ok = i0 + v < n;
#pragma unroll
                for (int c = 0; c < 4; ++c) s[c][v] = ok ? a.env.state[c * ld + i0 + v] : T(0);
                p[v] = ok ? load_xi(a.env.xi, i0 + v) : Xi<T>{ T(1), T(1), T(1), T(1) };
                el[v] = !ok ? 0 : kLean ? (int32_t)a.env.elapsed16[i0 + v] : a.env.elapsed[i0 + v];
                act[v] = ok ? a.action[i0 + v] : 0;
            }
        }

        T rew[V];
        uint8_t dn[V], tr[V];
        const bool euler = a.euler != 0;
        bool bad_action = false;            // Discrete(2).contains (:173-174): the host raises at its next sync
#pragma unroll
        for (int v = 0; v < V; ++v) {
            bad_action = bad_action || act[v] > 1;
            State<T> st = { s[0][v], s[1][v], s[2][v], s[3][v] };
            const bool terminated = dynamics(st, p[v], derive(p[v]), act[v], euler);
            s[0][v] = st.x; s[1][v] = st.x_dot; s[2][v] = st.theta; s[3][v] = st.theta_dot;
            el[v] += 1;                                                    // TimeLimit.step
            bool done = terminated, trunc = false;
            if (a.max_steps > 0 && el[v] >= a.max_steps) { trunc = !terminated; done = true; }
            T r = T(1);                                                    // :207-212
            if (!kAutoReset && i0 + v < n && terminated) {
                const int32_t b = a.env.beyond[i0 + v];                    // :213-222 (only reachable without auto-reset)
                a.env.beyond[i0 + v] = b < 0 ? 0 : b + 1;
                r = b < 0 ? T(1) : T(0);
            }
            rew[v] = r; dn[v] = done; tr[v] = trunc;
            if (kAutoReset && done && i0 + v < n) {
                const int32_t len = trunc ? -el[v] : el[v];
                el[v] = 0;
                if (kLog) {
                    const unsigned slot = atomicAdd(&s_count, 1u);
                    s_list[slot] = (uint16_t)(threadIdx.x * V + v);
                    s_len[slot] = len;
                } else {
                    s_list[atomicAdd(&s_count, 1u)] = (uint16_t)(threadIdx.x * V + v);
                }
            }
        }
        if (bad_action && a.counters) atomicAdd(a.counters + kCounterBadAction, 1ull);

        if (kNoisy) {       // obs = new state + std * N(0, I); a finished env's obs is overwritten by its reset below
            T o[4][V];
#pragma unroll
            for (int v = 0; v < V; ++v) {
                T ov[4];
                add_obs_noise(State<T>{ s[0][v], s[1][v], s[2][v], s[3][v] }, a.env.noise_std, a.env.seed,
                              a.env.env_id0 + (uint64_t)(i0 + v), a.tick, 0u, ov);
#pragma unroll
                for (int c = 0; c < 4; ++c) o[c][v] = ov[c];
            }
            if (full) {
#pragma unroll
                for (int c = 0; c < 4; ++c) vstore<typename VT::Real>(a.env.obs + c * ld + i0, o[c]);
            } else {
#pragma unroll
                for (int v = 0; v < V; ++v)
                    if (i0 + v < n) {
#pragma unroll
                        for (int c = 0; c < 4; ++c) a.env.obs[c * ld + i0 + v] = o[c][v];
                    }
            }
        }

        // (a): trigger AFTER the arithmetic: the dependent grid becomes launchable when every CTA of this one is about
        // to store, so its CTAs spin in griddepcontrol.wait only briefly.  Triggering at kernel entry was 4 % faster
        // for one stream but cost 4 independent graph branches 1 % (round 1).
        if (!tracked) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
        if (full) {
#pragma unroll
            for (int c = 0; c < 4; ++c) vstore<typename VT::Real>(a.env.state + c * ld + i0, s[c]);
            if (kLean) {
                uint16_t e16[V];
#pragma unroll
                for (int v = 0; v < V; ++v) e16[v] = (uint16_t)el[v];
                vstore<typename VT::Half>(a.env.elapsed16 + i0, e16);
            } else {
                vstore<typename VT::Int>(a.env.elapsed + i0, el);
            }
            if (a.reward) vstore<typename VT::Real>(a.reward + i0, rew);
            vstore<typename VT::Byte>(a.done + i0, dn);
            if (a.truncated) vstore<typename VT::Byte>(a.truncated + i0, tr);
        } else {
#pragma unroll
            for (int v = 0; v < V; ++v) {
                if (i0 + v < n) {
#pragma unroll
                    for (int c = 0; c < 4; ++c) a.env.state[c * ld + i0 + v] = s[c][v];
                    if (kLean) a.env.elapsed16[i0 + v] = (uint16_t)el[v];
                    else a.env.elapsed[i0 + v] = el[v];
                    if (a.reward) a.reward[i0 + v] = rew[v];
                    a.done[i0 + v] = dn[v];
                    if (a.truncated) a.truncated[i0 + v] = tr[v];
                }
            }
        }
    } else if (!tracked) {
        asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
    }

    if (kAutoReset) {
        __syncthreads();                    // list complete; the owners' stores above are ordered before ours
        const unsigned count = s_count;
        unsigned viol = 0;
        for (unsigned j = threadIdx.x; j < count; j += kStepThreads) {
            if (kLog) {
                const int64_t i = block0 + s_list[j];
                const int32_t len = s_len[j];
                const State<T> fs = { a.env.state[i], a.env.state[ld + i], a.env.state[2 * ld + i], a.env.state[3 * ld + i] };
                const uint32_t c = (uint32_t)log.count[i];
                log_episode(log, ld, i, c, load_xi(a.env.xi, i), fs, len < 0 ? -len : len, len < 0, a.tick);
                log.count[i] = (int32_t)(c + 1u);
            }
            if (kScen) {        // env i's scenario row, read here only (through L1: few distinct rows per CTA)
                const int64_t i = block0 + s_list[j];
                viol += reset_env<T, true>(a.env, scenario_row<T>(env_scen.rows, env_scenario(env_scen, i)), i, a.tick,
                                           a.env.seed);
            } else if (kMix) {  // the drawn row: one more Philox block and one 8-byte table load per reset
                const int64_t i = block0 + s_list[j];
                const uint32_t c = mixture_draw(mix, a.env.seed, a.env.env_id0 + (uint64_t)i, a.tick);
                viol += reset_env<T, true>(a.env, scenario_row<T>(mix.rows, c), i, a.tick, a.env.seed);
                mix.of_env[i] = (uint16_t)c;
            } else {
                viol += reset_env(a.env, a.dr, block0 + s_list[j], a.tick, a.env.seed);
            }
        }
        if (viol && a.counters) atomicAdd(a.counters + kCounterGaussian, (unsigned long long)viol);
    }
    if (tracked) {
        __syncthreads();                    // every store of the CTA precedes (happens-before) thread 0's release
        if (threadIdx.x == 0) {
            st_release_gpu(a.env.progress + 2 * (size_t)blockIdx.x + 1, (kScen || kMix ? s_ticket : ticket) + 1u);
            asm volatile("griddepcontrol.wait;" ::: "memory");     // do not complete before the previous grid has
        }
    }
