// C ABI of librenv_b200.so (declared in include/renv.h): argument validation + kernel launches.
// Stateless and re-entrant: nothing is allocated, cached or synchronised here.
#include "../../include/renv.h"
#include "renv_kernels.cuh"
#include <cmath>
#include "renv_rollout_pair.cuh"
#include "renv_fullgauss_tc.cuh"
#include "renv_mlp_policy.cuh"
#include "renv_mlp_gae.cuh"
#include "renv_transition_loglik.cuh"
#include "renv_scalar_server.cuh"
#include <stddef.h>
#include <stdlib.h>
#include <string.h>
#include <type_traits>

using namespace renv;

namespace {

inline bool aligned(const void *p, size_t a) { return (reinterpret_cast<uintptr_t>(p) & (a - 1)) == 0; }

// Host-side conversion of the 4-dim DR configuration to the kernels' element type: the same casts, the same
// rounded-once `hi - lo` and the exact 2^-24 folding the device code used to do per reset.
template <typename T> int to_cfg4(const renv_dr_cfg *dr, DrCfg4<T> *out)
{
    out->dr_type = kDrNone;
    out->dim = 4;
    for (int k = 0; k < 4; ++k) { out->a[k] = T(0); out->b[k] = T(0); out->floor[k] = T(0); }
    for (int k = 0; k < 16; ++k) out->factor[k] = T(0);
    if (dr == nullptr || dr->dr_type == RENV_DR_NONE) return RENV_OK;
    if (dr->dr_type < RENV_DR_NONE || dr->dr_type > RENV_DR_FULLGAUSSIAN) return RENV_E_DRTYPE;
    if (dr->dim != 4) return RENV_E_DIM;
    out->dr_type = dr->dr_type;
    for (int k = 0; k < 4; ++k) {
        const T a = (T)dr->a[k], b = (T)dr->b[k];
        out->a[k] = a;
        if (dr->dr_type == RENV_DR_UNIFORM) {
            const T width = b - a;
            out->b[k] = sizeof(T) == 4 ? (T)(width * (T)(1.0 / 16777216.0)) : width;
            out->floor[k] = T(0);
        } else if (dr->dr_type == RENV_DR_FULLGAUSSIAN) {
            out->b[k] = b;                       // search-bound lo
            out->floor[k] = (T)dr->lb[k];        // search-bound hi
        } else {
            out->b[k] = b;
            out->floor[k] = dr->dr_type == RENV_DR_TRUNCNORM ? (T)dr->lb[k] : (T)0.1;
        }
    }
    if (dr->dr_type == RENV_DR_FULLGAUSSIAN)
        for (int k = 0; k < 16; ++k) out->factor[k] = (T)dr->factor[k];
    return RENV_OK;
}

enum ElapsedKind { kNeedElapsed32, kNeedElapsed16, kNeedEitherElapsed };
// kNeedEitherElapsed: the kernels take the int32 counter when env->elapsed is set, else the uint16 one.
template <typename T>
int check_env(const renv_cartpole_env *env, bool need_beyond, EnvPtrs<T> *out, ElapsedKind elapsed = kNeedElapsed32)
{
    if (env == nullptr || env->state == nullptr || env->xi == nullptr) return RENV_E_NULL;
    if (elapsed == kNeedElapsed32 && env->elapsed == nullptr) return RENV_E_NULL;
    if (elapsed == kNeedElapsed16 && env->elapsed16 == nullptr) return RENV_E_NULL;
    if (elapsed == kNeedEitherElapsed && env->elapsed == nullptr && env->elapsed16 == nullptr) return RENV_E_NULL;
    if (need_beyond && env->beyond == nullptr) return RENV_E_NULL;
    if (env->n <= 0 || env->ld < env->n) return RENV_E_SIZE;
    constexpr int V = VecTraits<T>::V;
    if (env->ld % V != 0) return RENV_E_ALIGN;
    if (!aligned(env->state, 16) || !aligned(env->xi, 16) || !aligned(env->elapsed, 16) || !aligned(env->elapsed16, 16) ||
        (env->episode && !aligned(env->episode, 4)) || !aligned(env->progress, 8) || (env->beyond && !aligned(env->beyond, 4)))
        return RENV_E_ALIGN;
    out->state = static_cast<T *>(env->state);
    out->xi = static_cast<T *>(env->xi);
    out->elapsed = env->elapsed;
    out->elapsed16 = env->elapsed16;
    out->progress = env->progress;
    out->episode = env->episode;
    out->beyond = env->beyond;
    out->n = env->n;
    out->ld = env->ld;
    out->env_id0 = env->env_id0;
    out->seed = env->seed;
    out->obs = nullptr;
    out->noise_std = T(0);
    return RENV_OK;
}

// "Noisy" variants: attach the observation buffer.  noise == nullptr: plain env (obs is the state itself).
template <typename T> int attach_noise(const renv_obs_noise *noise, EnvPtrs<T> *env)
{
    if (noise == nullptr) return RENV_OK;
    if (noise->obs == nullptr) return RENV_E_NULL;
    if (!aligned(noise->obs, 16)) return RENV_E_ALIGN;
    if (!(noise->std >= 0.0)) return RENV_E_ARG;
    env->obs = static_cast<T *>(noise->obs);
    env->noise_std = (T)noise->std;
    return RENV_OK;
}

template <typename T> int check_log(const renv_episode_log *log, LogPtrs<T> *out)
{
    if (log == nullptr || log->xi == nullptr || log->final_state == nullptr || log->length == nullptr ||
        log->truncated == nullptr || log->end_tick == nullptr || log->count == nullptr)
        return RENV_E_NULL;
    if (log->capacity < 1 || log->capacity > 0x7fffffffLL) return RENV_E_SIZE;
    if (!aligned(log->xi, 16) || !aligned(log->final_state, 16) || !aligned(log->length, 4) || !aligned(log->end_tick, 8) ||
        !aligned(log->count, 4))
        return RENV_E_ALIGN;
    out->xi = static_cast<T *>(log->xi);
    out->final_state = static_cast<T *>(log->final_state);
    out->length = log->length;
    out->truncated = log->truncated;
    out->end_tick = log->end_tick;
    out->count = log->count;
    out->capacity = (uint32_t)log->capacity;
    return RENV_OK;
}

inline int launch_status() { return (int)cudaGetLastError(); }

// Blocks of `per_block` items each for n items; RENV_E_SIZE when the grid does not fit in a launch.
inline int grid_for(int64_t n, int64_t per_block, unsigned *blocks)
{
    const int64_t g = (n + per_block - 1) / per_block;
    if (g > 0x7fffffffLL) return RENV_E_SIZE;
    *blocks = (unsigned)g;
    return RENV_OK;
}

int sm_count(int *sms)
{
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(sms, cudaDevAttrMultiProcessorCount, dev);
    return (int)e;
}

// One wave of persistent CTAs over tiles of `per_cta` items: min(tiles, SMs x ctas_per_sm).
int persistent_grid(int64_t n, int per_cta, int ctas_per_sm, unsigned *grid)
{
    int sms = 0;
    const int rc = sm_count(&sms);
    if (rc) return rc;
    const int64_t tiles = (n + per_cta - 1) / per_cta;
    *grid = (unsigned)(tiles < (int64_t)sms * ctas_per_sm ? tiles : (int64_t)sms * ctas_per_sm);
    return RENV_OK;
}

// A runtime choice as a template argument: f(std::integral_constant<...>{}) for the value given.
template <typename F> void with_flag(bool b, F &&f)
{
    if (b) f(std::true_type{});
    else f(std::false_type{});
}
template <typename F> void with_activation(int activation, F &&f)
{
    if (activation == RENV_MLP_TANH) f(std::integral_constant<int, kMlpTanh>{});
    else f(std::integral_constant<int, kMlpRelu>{});
}
// The 8 instances of the MLP rollout and collect kernels: f(activation, euler, logged).
template <typename F> void with_mlp_instance(int activation, bool euler, bool logged, F &&f)
{
    with_activation(activation, [&](auto act) {
        with_flag(euler, [&](auto eu) { with_flag(logged, [&](auto lg) { f(act, eu, lg); }); });
    });
}

// Launch with programmatic stream serialization: the kernel may start while its predecessor in the stream drains and
// synchronises itself with griddepcontrol.wait (see cartpole_step_kernel).  Captured into CUDA graphs as a
// programmatic dependency edge.
template <typename Args>
int launch_pdl(void (*kernel)(const Args), unsigned blocks, unsigned threads, cudaStream_t stream, const Args &args)
{
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = dim3(blocks, 1, 1);
    cfg.blockDim = dim3(threads, 1, 1);
    cfg.dynamicSmemBytes = 0;
    cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    const cudaError_t rc = cudaLaunchKernelEx(&cfg, kernel, args);
    return rc != cudaSuccess ? (int)rc : launch_status();
}

// fp32: the packed-transform kernel; fp64: the generic one
template <int kType, int kStore>
void launch_sampler(float *out, int64_t n, const DrCfgPrepared<float> &c, uint64_t seed, uint64_t sample_id0, uint32_t call,
                    unsigned long long *violations, int items, unsigned blocks, cudaStream_t st)
{
    const PhiloxKeys ks = philox_keys((uint32_t)seed, (uint32_t)(seed >> 32));
    dr_sample_f32_kernel<kType, kStore><<<blocks, kSampleThreads, 0, st>>>(out, n, c, seed, ks, sample_id0, call, violations, items);
}
template <int kType, int kStore>
void launch_sampler(double *out, int64_t n, const DrCfgPrepared<double> &c, uint64_t seed, uint64_t sample_id0, uint32_t call,
                    unsigned long long *violations, int items, unsigned blocks, cudaStream_t st)
{
    if (kType == kDrUniform) {
        // the fast loop pre-scales the widths by 2^-53: exact unless a width is subnormal-small or not finite
        bool plain = true;
        for (int k = 0; k < c.dim; ++k) plain = plain && (c.b[k] == 0.0 || (std::fabs(c.b[k]) > 1e-250 && std::isfinite(c.b[k])));
        if (plain) {
            const PhiloxKeys ks = philox_keys((uint32_t)seed, (uint32_t)(seed >> 32));
            dr_sample_f64_uniform_kernel<kStore><<<blocks, kSampleThreads, 0, st>>>(out, n, c, ks, sample_id0, call, items);
            return;
        }
    }
    dr_sample_kernel<double, kType, kStore><<<blocks, kSampleThreads, 0, st>>>(out, n, c, seed, sample_id0, call, violations, items);
}

// fullgaussian, fp32, 17 <= dim <= 32: the tcgen05 kernel (renv_fullgauss_tc.cuh), one wave of persistent CTAs.
// Returns false when the tensor path does not apply (fp64, or switched off for A/B tests) and the caller falls through
// to the CUDA-core kernel.
bool launch_fullgaussian_tc(double *, int64_t, const FullGaussCfg<double> &, uint64_t, uint64_t, uint32_t,
                            unsigned long long *, cudaStream_t, int *) { return false; }
bool launch_fullgaussian_tc(float *out, int64_t n, const FullGaussCfg<float> &g, uint64_t seed, uint64_t sample_id0,
                            uint32_t call, unsigned long long *counters, cudaStream_t st, int *rc)
{
    const char *knob = getenv("RENV_FULLGAUSS_TENSOR");           // "0": CUDA-core kernel (tests compare the two)
    if (knob && knob[0] == '0') return false;
    unsigned grid = 0;
    if ((*rc = persistent_grid(n, kFgTile, kFgCtas, &grid))) return true;
    FullGaussCfg<float> gt = g;
    for (int k = 0; k < 32; ++k) {      // the kernel's epilogue takes the WIDTH hi - lo (rounded once, as denormalize does) and mean / 4 (exact)
        gt.hi[k] = g.hi[k] - g.lo[k];
        gt.mean[k] = 0.25f * g.mean[k];
    }
    const PhiloxKeys ks = philox_keys((uint32_t)seed, (uint32_t)(seed >> 32));
    dr_sample_fullgaussian_tc_kernel<<<grid, kFgThreads, 0, st>>>(out, n, gt, ks, sample_id0, call, counters);
    *rc = launch_status();
    return true;
}

template <typename T>
int dr_sample(T *out, int64_t n, const renv_dr_cfg *cfg, uint64_t seed, uint64_t sample_id0, uint32_t call,
              unsigned long long *violations, void *stream)
{
    int rc_tc = RENV_OK;
    if (out == nullptr || cfg == nullptr) return RENV_E_NULL;
    if (n <= 0) return RENV_E_SIZE;
    if (cfg->dim < 1 || cfg->dim > RENV_MAX_DIM) return RENV_E_DIM;
    if (cfg->dr_type < RENV_DR_UNIFORM || cfg->dr_type > RENV_DR_FULLGAUSSIAN) return RENV_E_DRTYPE;
    if (!aligned(out, 16)) return RENV_E_ALIGN;
    if (cfg->dr_type == RENV_DR_FULLGAUSSIAN) {
        FullGaussCfg<T> g;
        g.dim = cfg->dim;
        for (int k = 0; k < 32; ++k) {
            const bool ok = k < cfg->dim;
            g.mean[k] = ok ? (T)cfg->a[k] : T(0); g.lo[k] = ok ? (T)cfg->b[k] : T(0); g.hi[k] = ok ? (T)cfg->lb[k] : T(0);
        }
        for (int k = 0; k < 32; ++k)                 // transposed, zero-padded: ft[k][d] = F[d][k]
            for (int d = 0; d < 32; ++d)
                g.ft[k * 32 + d] = (k < cfg->dim && d < cfg->dim) ? (T)cfg->factor[d * cfg->dim + k] : T(0);
        unsigned gblocks = 0;
        if (const int rc = grid_for(n, kFullGaussThreads, &gblocks)) return rc;
        const cudaStream_t gst = static_cast<cudaStream_t>(stream);
        if (cfg->dim > 16 && launch_fullgaussian_tc(out, n, g, seed, sample_id0, call, violations, gst, &rc_tc)) return rc_tc;
        if (cfg->dim <= 4) dr_sample_fullgaussian_kernel<T, 4><<<gblocks, kFullGaussThreads, 0, gst>>>(out, n, g, seed, sample_id0, call);
        else if (cfg->dim <= 8) dr_sample_fullgaussian_kernel<T, 8><<<gblocks, kFullGaussThreads, 0, gst>>>(out, n, g, seed, sample_id0, call);
        else if (cfg->dim <= 16) dr_sample_fullgaussian_kernel<T, 16><<<gblocks, kFullGaussThreads, 0, gst>>>(out, n, g, seed, sample_id0, call);
        else dr_sample_fullgaussian_kernel<T, 32><<<gblocks, kFullGaussThreads, 0, gst>>>(out, n, g, seed, sample_id0, call);
        return launch_status();
    }
    // host-side image of renv_dr.cuh load_dim_block: same conversions, same order, done once per launch
    DrCfgPrepared<T> c;
    c.dr_type = cfg->dr_type;
    c.dim = cfg->dim;
    for (int k = 0; k < 32; ++k) {
        const bool ok = k < cfg->dim;
        const T a = ok ? (T)cfg->a[k] : T(0), b = ok ? (T)cfg->b[k] : T(0);
        c.a[k] = a;
        if (cfg->dr_type == RENV_DR_UNIFORM) {
            const T width = b - a;                                          // rounded once, as numpy's `high - low`
            c.b[k] = sizeof(T) == 4 ? (T)(width * (T)(1.0 / 16777216.0)) : (T)width;   // fp32: 2^-24 folded in (exact)
        } else {
            c.b[k] = b;
        }
        c.floor[k] = !ok ? T(0) : cfg->dr_type == RENV_DR_TRUNCNORM ? (T)cfg->lb[k] : (T)0.1;
    }
    const int items = sampler_items<T>(n, cfg->dim);
    const int kTile = tile_samples<T>(cfg->dim, items);
    unsigned blocks = 0;
    if (const int rc = grid_for(n, kTile, &blocks)) return rc;
    // store width follows the row alignment: whole 128-bit blocks, float pairs (e.g. the 30-dim humanoid), scalars
    constexpr int P = Pack<T>::kPerBlock;
    const int store = cfg->dim % P == 0 ? 0 : (sizeof(T) == 4 && cfg->dim % 2 == 0 ? 1 : 2);
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
#define RENV_LAUNCH_SAMPLER(TYPE, STORE) launch_sampler<TYPE, STORE>(out, n, c, seed, sample_id0, call, violations, items, blocks, st)
#define RENV_LAUNCH_SAMPLER_TYPE(TYPE) \
    do { if (store == 0) RENV_LAUNCH_SAMPLER(TYPE, 0); else if (store == 1) RENV_LAUNCH_SAMPLER(TYPE, 1); \
         else RENV_LAUNCH_SAMPLER(TYPE, 2); } while (0)
    if (cfg->dr_type == RENV_DR_UNIFORM) RENV_LAUNCH_SAMPLER_TYPE(kDrUniform);
    else if (cfg->dr_type == RENV_DR_TRUNCNORM) RENV_LAUNCH_SAMPLER_TYPE(kDrTruncnorm);
    else RENV_LAUNCH_SAMPLER_TYPE(kDrGaussian);
#undef RENV_LAUNCH_SAMPLER_TYPE
#undef RENV_LAUNCH_SAMPLER
    return launch_status();
}

template <typename T>
int cartpole_reset(const renv_cartpole_env *env, const renv_obs_noise *noise, const uint8_t *mask, uint64_t tick,
                   const renv_dr_cfg *dr, unsigned long long *violations, void *stream)
{
    ResetArgs<T> a;
    int rc = check_env<T>(env, false, &a.env, kNeedEitherElapsed);
    if (rc) return rc;
    rc = attach_noise<T>(noise, &a.env);
    if (rc) return rc;
    rc = to_cfg4<T>(dr, &a.dr);
    if (rc) return rc;
    a.mask = mask;
    a.tick = tick;
    a.violations = violations;
    unsigned blocks = 0;
    if ((rc = grid_for(env->n, 256, &blocks))) return rc;
    cartpole_reset_kernel<T><<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(a);
    return launch_status();
}

// A step CTA covers one tile of envs, the granule of renv_cartpole_env.progress: callers size that array from the
// header's tile sizes, so the kernels must use the same ones.
static_assert(kStepThreads * VecTraits<float>::V == RENV_TILE_ENVS_F32, "fp32 step tile differs from include/renv.h");
static_assert(kStepThreads * VecTraits<double>::V == RENV_TILE_ENVS_F64, "fp64 step tile differs from include/renv.h");

template <typename T, bool kLean>
int cartpole_step(const renv_cartpole_env *env, const renv_obs_noise *noise, const uint8_t *action, T *reward,
                  uint8_t *done, uint8_t *truncated, int integrator, int max_steps, int auto_reset, uint64_t tick,
                  const renv_dr_cfg *dr, unsigned long long *counters, void *stream,
                  const renv_episode_log *log = nullptr, bool logged = false)
{
    StepArgs<T> a;
    const ElapsedKind counter = kLean ? kNeedElapsed16 : logged && sizeof(T) == 4 ? kNeedEitherElapsed : kNeedElapsed32;
    int rc = check_env<T>(env, !auto_reset, &a.env, counter);
    if (rc) return rc;
    rc = attach_noise<T>(noise, &a.env);
    if (rc) return rc;
    LoggedStepArgs<T> la;
    if (logged && (rc = check_log<T>(log, &la.log))) return rc;
    if (action == nullptr || done == nullptr) return RENV_E_NULL;
    if (reward == nullptr && !auto_reset) return RENV_E_NULL;      // only the auto-reset reward is the constant 1.0
    if (!aligned(action, 4) || !aligned(reward, 16) || !aligned(done, 4) || (truncated && !aligned(truncated, 4)))
        return RENV_E_ALIGN;
    if (counters && !aligned(counters, 8)) return RENV_E_ALIGN;
    if (integrator != RENV_EULER && integrator != RENV_SEMI_IMPLICIT) return RENV_E_INTEGRATOR;
    if ((kLean || env->elapsed == nullptr) && max_steps > 65535) return RENV_E_SIZE;
    rc = to_cfg4<T>(auto_reset ? dr : nullptr, &a.dr);
    if (rc) return rc;
    a.action = action; a.reward = reward; a.done = done; a.truncated = truncated;
    a.euler = integrator == RENV_EULER;
    a.max_steps = max_steps;
    a.tick = tick;
    a.counters = counters;
    unsigned blocks = 0;
    if ((rc = grid_for(env->n, (int64_t)kStepThreads * VecTraits<T>::V, &blocks))) return rc;
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    const bool noisy = a.env.obs != nullptr;
    if (logged) {
        la.step = a;
        return launch_pdl(cartpole_step_logged_kernel<T>, blocks, kStepThreads, st, la);
    }
    if (kLean) return launch_pdl(cartpole_step_kernel<T, true, false, true>, blocks, kStepThreads, st, a);
    if (auto_reset && !noisy) return launch_pdl(cartpole_step_kernel<T, true, false>, blocks, kStepThreads, st, a);
    if (auto_reset) return launch_pdl(cartpole_step_kernel<T, true, true>, blocks, kStepThreads, st, a);
    if (!noisy) return launch_pdl(cartpole_step_kernel<T, false, false>, blocks, kStepThreads, st, a);
    return launch_pdl(cartpole_step_kernel<T, false, true>, blocks, kStepThreads, st, a);
}

// The checks and arguments every fused rollout shares (linear policy, MLP policy, collect), after the caller's checks
// of the env, the log, the policy and stats == NULL (the linear rollout checks its policy between that and the
// alignment of stats).
template <typename T>
int check_rollout(double *stats, int K, int integrator, int max_steps, uint64_t tick, const renv_dr_cfg *dr,
                  unsigned long long *violations, const Policy<T> &policy, RolloutArgs<T> *a)
{
    if (!aligned(stats, 8)) return RENV_E_ALIGN;
    if (K <= 0 || K > (1 << 30)) return RENV_E_SIZE;      // per-thread step counters are 32-bit
    if (integrator != RENV_EULER && integrator != RENV_SEMI_IMPLICIT) return RENV_E_INTEGRATOR;
    const int rc = to_cfg4<T>(dr, &a->dr);
    if (rc) return rc;
    a->policy = policy;
    a->K = K;
    a->euler = integrator == RENV_EULER;
    a->max_steps = max_steps;
    a->tick = tick;
    a->stats = stats;
    a->violations = violations;
    return RENV_OK;
}

// The linear-policy rollout kernels (la.log is read only when logged).  One env per thread, except the fp32 linear
// policy on the true state: an env PAIR per thread on the packed FFMA2 pipe (renv_rollout_pair.cuh).  The random
// policy keeps one env per thread for both element types (an env draws one Philox block per 128 env-steps for its
// action bits): the pair kernel was tried for it and is slower (1.4e11 vs 2.4e11 env-steps/s at the time, 3.2e11
// now), because with ~27-step episodes a pair spends most packed steps with one slot parked for its reset.
template <typename T> int launch_rollout(const LoggedRolloutArgs<T> &la, bool logged, bool random, cudaStream_t st)
{
    const RolloutArgs<T> &a = la.roll;
    const bool noisy = a.env.obs != nullptr;
    const bool pair = std::is_same<T, float>::value && !random && !noisy;
    unsigned blocks = 0;
    const int rc = grid_for(pair ? (a.env.n + kPairSlots - 1) / kPairSlots : a.env.n, kRolloutThreads, &blocks);
    if (rc) return rc;
    with_flag(a.euler, [&](auto euler) {
        if (random) {
            if (logged) cartpole_rollout_logged_kernel<T, euler, true><<<blocks, kRolloutThreads, 0, st>>>(la);
            else cartpole_rollout_kernel<T, euler, false, true><<<blocks, kRolloutThreads, 0, st>>>(a);
        } else if (noisy) {       // the logged entry points take no noise block
            cartpole_rollout_kernel<T, euler, true><<<blocks, kRolloutThreads, 0, st>>>(a);
        } else if constexpr (std::is_same<T, float>::value) {
            if (logged) cartpole_rollout_pair_logged_kernel<euler><<<blocks, kRolloutThreads, 0, st>>>(la);
            else cartpole_rollout_pair_kernel<euler><<<blocks, kRolloutThreads, 0, st>>>(a);
        } else {
            if (logged) cartpole_rollout_logged_kernel<T, euler, false><<<blocks, kRolloutThreads, 0, st>>>(la);
            else cartpole_rollout_kernel<T, euler><<<blocks, kRolloutThreads, 0, st>>>(a);
        }
    });
    return launch_status();
}

template <typename T>
int cartpole_rollout(const renv_cartpole_env *env, const renv_obs_noise *noise, const double w[4], double b, int K,
                     int integrator, int max_steps, uint64_t tick, const renv_dr_cfg *dr, double *stats,
                     unsigned long long *violations, void *stream, const renv_episode_log *log = nullptr,
                     bool logged = false)
{
    LoggedRolloutArgs<T> la;
    int rc = check_env<T>(env, false, &la.roll.env, sizeof(T) == 4 ? kNeedEitherElapsed : kNeedElapsed32);
    if (rc) return rc;
    rc = attach_noise<T>(noise, &la.roll.env);
    if (rc) return rc;
    if (logged && (rc = check_log<T>(log, &la.log))) return rc;
    if (stats == nullptr) return RENV_E_NULL;
    if (w == nullptr && noise != nullptr) return RENV_E_ARG;      // the random policy does not look at observations
    const Policy<T> policy = w ? Policy<T>{ (T)w[0], (T)w[1], (T)w[2], (T)w[3], (T)b } : Policy<T>{ T(0), T(0), T(0), T(0), T(0) };
    rc = check_rollout<T>(stats, K, integrator, max_steps, tick, dr, violations, policy, &la.roll);
    if (rc) return rc;
    if (env->elapsed == nullptr && max_steps > 65535) return RENV_E_SIZE;     // the uint16 counter
    return launch_rollout(la, logged, w == nullptr, static_cast<cudaStream_t>(stream));
}

// MLP policy (renv_mlp_policy.cuh): the packed parameters and the activation.
int check_mlp(const renv_mlp_policy *p)
{
    if (p == nullptr || p->params == nullptr) return RENV_E_NULL;
    if (!aligned(p->params, 16)) return RENV_E_ALIGN;
    if (p->activation != RENV_MLP_TANH && p->activation != RENV_MLP_RELU) return RENV_E_ARG;
    return RENV_OK;
}

// renv_cartpole_policy_logp_mlp_f32 (with_logp) and renv_cartpole_policy_actions_mlp_f32 (argmax only: sample 0, no
// logp), each on its own kernel.
int policy_mlp(const renv_cartpole_env *env, const renv_mlp_policy *p, bool with_logp, int sample, uint64_t tick,
               uint8_t *action, float *logp, float *logits, void *stream)
{
    if (env == nullptr || env->state == nullptr) return RENV_E_NULL;
    int rc = check_mlp(p);
    if (rc) return rc;
    if (action == nullptr) return RENV_E_NULL;
    if (env->n <= 0 || env->ld < env->n) return RENV_E_SIZE;
    if (env->ld % 4 != 0 || !aligned(env->state, 16) || !aligned(action, 4) || !aligned(logits, 16) || !aligned(logp, 4))
        return RENV_E_ALIGN;
    if (sample != 0 && sample != 1) return RENV_E_ARG;
    MlpLogpArgs a;
    a.act.state = static_cast<const float *>(env->state);
    a.act.n = env->n; a.act.ld = env->ld;
    a.act.params = static_cast<const float *>(p->params);
    a.act.action = action; a.act.logits = logits;
    a.logp = logp;
    a.env_id0 = env->env_id0; a.seed = env->seed; a.tick = tick;
    a.sample = sample;
    unsigned grid = 0;
    if ((rc = persistent_grid(env->n, kMlpThreads, with_logp ? kMlpRolloutCtas : kMlpCtas, &grid))) return rc;
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    with_activation(p->activation, [&](auto act) {
        if (with_logp) cartpole_policy_logp_mlp_kernel<act><<<grid, kMlpThreads, 0, st>>>(a);
        else cartpole_policy_actions_mlp_kernel<act><<<grid, kMlpThreads, 0, st>>>(a.act);
    });
    return launch_status();
}

// The argument checks and arguments shared by the MLP rollout and collect entry points (A: MlpRolloutArgs or
// MlpCollectArgs).
template <typename A>
int prepare_rollout_mlp(const renv_cartpole_env *env, const renv_episode_log *log, bool logged, const renv_mlp_policy *p,
                        int K, int integrator, int max_steps, uint64_t tick, const renv_dr_cfg *dr, double *stats,
                        unsigned long long *violations, A *a, unsigned *blocks)
{
    int rc = check_env<float>(env, false, &a->roll.env, kNeedEitherElapsed);
    if (rc) return rc;
    if (logged && (rc = check_log<float>(log, &a->log))) return rc;
    if (!logged) a->log = LogPtrs<float>{};
    if ((rc = check_mlp(p))) return rc;
    if (stats == nullptr) return RENV_E_NULL;
    const Policy<float> unused{ 0.0f, 0.0f, 0.0f, 0.0f, 0.0f };
    if ((rc = check_rollout<float>(stats, K, integrator, max_steps, tick, dr, violations, unused, &a->roll))) return rc;
    if (env->elapsed == nullptr && max_steps > 65535) return RENV_E_SIZE;     // the uint16 counter
    a->params = static_cast<const float *>(p->params);
    return grid_for(env->n, kMlpThreads, blocks);
}

int rollout_mlp(const renv_cartpole_env *env, const renv_episode_log *log, bool logged, const renv_mlp_policy *p, int K,
                int integrator, int max_steps, uint64_t tick, const renv_dr_cfg *dr, double *stats,
                unsigned long long *violations, void *stream)
{
    MlpRolloutArgs a;
    unsigned blocks = 0;
    const int rc = prepare_rollout_mlp(env, log, logged, p, K, integrator, max_steps, tick, dr, stats, violations, &a, &blocks);
    if (rc) return rc;
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    with_mlp_instance(p->activation, a.roll.euler, logged, [&](auto act, auto euler, auto lg) {
        cartpole_rollout_mlp_kernel<act, euler, lg><<<blocks, kMlpThreads, 0, st>>>(a);
    });
    return launch_status();
}

int check_traj(const renv_trajectory *t, int K, MlpTrajPtrs *out)
{
    if (t == nullptr || t->obs == nullptr || t->action == nullptr || t->done == nullptr) return RENV_E_NULL;
    if (!aligned(t->obs, 16) || !aligned(t->final_obs, 16) || !aligned(t->action, 4) || !aligned(t->done, 4) ||
        !aligned(t->logp, 4) || !aligned(t->truncated, 4))
        return RENV_E_ALIGN;
    if (K > t->capacity) return RENV_E_ARG;
    *out = MlpTrajPtrs{ t->obs, t->action, t->done, t->logp, t->truncated, t->final_obs };
    return RENV_OK;
}

int collect_mlp(const renv_cartpole_env *env, const renv_episode_log *log, bool logged, const renv_mlp_policy *p,
                const renv_trajectory *traj, int sample, int K, int integrator, int max_steps, uint64_t tick,
                const renv_dr_cfg *dr, double *stats, unsigned long long *violations, void *stream)
{
    MlpCollectArgs a;
    unsigned blocks = 0;
    int rc = prepare_rollout_mlp(env, log, logged, p, K, integrator, max_steps, tick, dr, stats, violations, &a, &blocks);
    if (rc) return rc;
    if ((rc = check_traj(traj, K, &a.traj))) return rc;
    if (sample != 0 && sample != 1) return RENV_E_ARG;
    a.sample = sample;
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    with_mlp_instance(p->activation, a.roll.euler, logged, [&](auto act, auto euler, auto lg) {
        cartpole_collect_mlp_kernel<act, euler, lg><<<blocks, kMlpThreads, 0, st>>>(a);
    });
    return launch_status();
}

int gae_mlp(const renv_cartpole_env *env, const renv_mlp_policy *critic, const renv_trajectory *traj, int K, float gamma,
            float lambda, float *values, float *advantages, float *returns, void *stream)
{
    if (env == nullptr || env->state == nullptr) return RENV_E_NULL;
    int rc = check_mlp(critic);
    if (rc) return rc;
    if (traj == nullptr || traj->obs == nullptr || traj->done == nullptr || traj->truncated == nullptr ||
        traj->final_obs == nullptr || values == nullptr || advantages == nullptr || returns == nullptr)
        return RENV_E_NULL;
    if (env->n <= 0 || env->ld < env->n) return RENV_E_SIZE;
    if (env->ld % 4 != 0 || !aligned(env->state, 16) || !aligned(traj->obs, 16) || !aligned(traj->final_obs, 16) ||
        !aligned(traj->done, 4) || !aligned(traj->truncated, 4) || !aligned(values, 4) || !aligned(advantages, 4) ||
        !aligned(returns, 4))
        return RENV_E_ALIGN;
    if (K <= 0) return RENV_E_SIZE;
    if (K > traj->capacity) return RENV_E_ARG;
    if (!(gamma >= 0.0f && gamma <= 1.0f) || !(lambda >= 0.0f && lambda <= 1.0f)) return RENV_E_ARG;   // NaN fails too
    unsigned blocks = 0;
    if ((rc = grid_for(env->n, kMlpThreads, &blocks))) return rc;
    MlpGaeArgs a;
    a.state = static_cast<const float *>(env->state);
    a.n = env->n; a.ld = env->ld;
    a.params = static_cast<const float *>(critic->params);
    a.obs = traj->obs; a.final_obs = traj->final_obs;
    a.done = traj->done; a.truncated = traj->truncated;
    a.values = values; a.advantages = advantages; a.returns = returns;
    a.K = K; a.gamma = gamma; a.lambda = lambda;
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    with_activation(critic->activation, [&](auto act) {
        cartpole_gae_mlp_kernel<act><<<blocks, kMlpThreads, 0, st>>>(a);
    });
    return launch_status();
}

// The checks and arguments both population entry points share, all before any CUDA call.  Only env->n, env_id0, seed
// and, without an active DR config, xi are read.  `rows` holds the P policy rows, aligned to `row_align` bytes.  The
// kernels start every episode at `tick` and step at tick + 1 .. tick + K (a->tick = tick + 1).
int prepare_population(const renv_cartpole_env *env, const void *rows, size_t row_align, int P, int K, int integrator,
                       int max_steps, uint64_t tick, const renv_dr_cfg *dr, double *stats,
                       unsigned long long *violations, RolloutArgs<float> *a, PopulationPtrs *pop)
{
    if (env == nullptr || rows == nullptr || stats == nullptr) return RENV_E_NULL;
    // P n < 2^31: the flat (member, env) index and the MLP grid fit in 31 bits
    if (P < 1 || env->n <= 0 || env->n >= (1LL << 31) || (int64_t)P * env->n >= (1LL << 31)) return RENV_E_SIZE;
    const Policy<float> unused{ 0.0f, 0.0f, 0.0f, 0.0f, 0.0f };
    const int rc = check_rollout<float>(stats, K, integrator, max_steps, tick + 1, dr, violations, unused, a);
    if (rc) return rc;
    const bool table = a->dr.dr_type == kDrNone;        // xi is row j of the env's table, else drawn at the fresh start
    if (table && env->xi == nullptr) return RENV_E_NULL;
    if ((table && !aligned(env->xi, 16)) || !aligned(rows, row_align)) return RENV_E_ALIGN;
    a->env = EnvPtrs<float>{};
    a->env.xi = table ? static_cast<float *>(env->xi) : nullptr;
    a->env.n = env->n;
    a->env.env_id0 = env->env_id0;
    a->env.seed = env->seed;
    *pop = PopulationPtrs{ static_cast<const float *>(rows), (int64_t)P * env->n,
                           (uint32_t)((env->n + kMlpThreads - 1) / kMlpThreads) };
    return RENV_OK;
}

int population_linear(const renv_cartpole_env *env, const float *policies, int P, int K, int integrator, int max_steps,
                      uint64_t tick, const renv_dr_cfg *dr, double *stats, unsigned long long *violations, void *stream)
{
    PopulationArgs pa;
    int rc = prepare_population(env, policies, 4, P, K, integrator, max_steps, tick, dr, stats, violations, &pa.roll, &pa.pop);
    if (rc) return rc;
    unsigned blocks = 0;
    if ((rc = grid_for(pa.pop.total, kRolloutThreads, &blocks))) return rc;
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    with_flag(pa.roll.euler, [&](auto euler) {
        cartpole_population_linear_kernel<euler><<<blocks, kRolloutThreads, 0, st>>>(pa);
    });
    return launch_status();
}

int population_mlp(const renv_cartpole_env *env, const void *params, int activation, int P, int K, int integrator,
                   int max_steps, uint64_t tick, const renv_dr_cfg *dr, double *stats, unsigned long long *violations,
                   void *stream)
{
    MlpPopulationArgs pa;
    const int rc = prepare_population(env, params, 16, P, K, integrator, max_steps, tick, dr, stats, violations,
                                      &pa.mlp.roll, &pa.pop);
    if (rc) return rc;
    if (activation != RENV_MLP_TANH && activation != RENV_MLP_RELU) return RENV_E_ARG;
    pa.mlp.params = nullptr;
    pa.mlp.log = LogPtrs<float>{};
    const unsigned blocks = (unsigned)P * pa.pop.ctas;      // <= P n < 2^31
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    with_activation(activation, [&](auto act) {
        with_flag(pa.mlp.roll.euler, [&](auto euler) {
            cartpole_population_mlp_kernel<act, euler><<<blocks, kMlpThreads, 0, st>>>(pa);
        });
    });
    return launch_status();
}

// A scenario row (include/renv.h RENV_SCENARIO_FLOATS) is the DrCfg4<float> image the kernels take, zero-padded.
static_assert(kScenarioFloats == RENV_SCENARIO_FLOATS, "scenario row size differs from include/renv.h");
static_assert(offsetof(DrCfg4<float>, dr_type) == 0 && offsetof(DrCfg4<float>, dim) == 4 &&
              offsetof(DrCfg4<float>, a) == 8 && offsetof(DrCfg4<float>, b) == 24 &&
              offsetof(DrCfg4<float>, floor) == 40 && offsetof(DrCfg4<float>, factor) == 56 &&
              sizeof(DrCfg4<float>) == 120, "scenario row layout differs from include/renv.h");

int scenario_pack(const renv_dr_cfg *dr, const double *task, float *out)
{
    if (out == nullptr) return RENV_E_NULL;
    DrCfg4<float> cfg;
    const int rc = to_cfg4<float>(dr, &cfg);
    if (rc) return rc;
    if (cfg.dr_type == kDrNone) {           // a fixed task: a = the task, kept across resets
        if (task == nullptr) return RENV_E_NULL;
        for (int k = 0; k < 4; ++k)
            if (!std::isfinite(task[k])) return RENV_E_ARG;
        for (int k = 0; k < 4; ++k) cfg.a[k] = (float)task[k];
    }
    float row[kScenarioFloats] = {};
    memcpy(row, &cfg, sizeof(cfg));
    memcpy(out, row, sizeof(row));
    return RENV_OK;
}

// The checks and arguments both grid entry points share, all before any CUDA call: those of a population launch on
// P C n (policy, scenario, env) triples, plus the scenario rows.  Neither env->xi nor a DR config is read.
int prepare_grid(const renv_cartpole_env *env, const void *rows, size_t row_align, int P, const float *scenarios, int C,
                 int K, int integrator, int max_steps, uint64_t tick, double *stats, unsigned long long *violations,
                 RolloutArgs<float> *a, PopulationPtrs *pop, GridPtrs *grid)
{
    if (env == nullptr || rows == nullptr || scenarios == nullptr || stats == nullptr) return RENV_E_NULL;
    // P C n < 2^31: the flat (policy, scenario, env) index, a member's (scenario, env) range and the MLP grid fit in 31 bits
    if (P < 1 || C < 1 || env->n <= 0 || env->n >= (1LL << 31) || (int64_t)P * C >= (1LL << 31) ||
        (int64_t)P * C * env->n >= (1LL << 31))
        return RENV_E_SIZE;
    const Policy<float> unused{ 0.0f, 0.0f, 0.0f, 0.0f, 0.0f };
    const int rc = check_rollout<float>(stats, K, integrator, max_steps, tick + 1, nullptr, violations, unused, a);
    if (rc) return rc;
    if (!aligned(rows, row_align) || !aligned(scenarios, 16)) return RENV_E_ALIGN;
    a->env = EnvPtrs<float>{};
    a->env.n = env->n;
    a->env.env_id0 = env->env_id0;
    a->env.seed = env->seed;
    const int64_t span = (int64_t)C * env->n;
    *pop = PopulationPtrs{ static_cast<const float *>(rows), (int64_t)P * span,
                           (uint32_t)((span + kMlpThreads - 1) / kMlpThreads) };
    *grid = GridPtrs{ scenarios, (uint32_t)C, (uint32_t)span };
    return RENV_OK;
}

int grid_linear(const renv_cartpole_env *env, const float *policies, int P, const float *scenarios, int C, int K,
                int integrator, int max_steps, uint64_t tick, double *stats, unsigned long long *violations, void *stream)
{
    GridArgs ga;
    int rc = prepare_grid(env, policies, 4, P, scenarios, C, K, integrator, max_steps, tick, stats, violations, &ga.roll,
                          &ga.pop, &ga.grid);
    if (rc) return rc;
    unsigned blocks = 0;
    if ((rc = grid_for(ga.pop.total, kRolloutThreads, &blocks))) return rc;
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    with_flag(ga.roll.euler, [&](auto euler) {
        cartpole_grid_linear_kernel<euler><<<blocks, kRolloutThreads, 0, st>>>(ga);
    });
    return launch_status();
}

int grid_mlp(const renv_cartpole_env *env, const void *params, int activation, int P, const float *scenarios, int C,
             int K, int integrator, int max_steps, uint64_t tick, double *stats, unsigned long long *violations,
             void *stream)
{
    MlpGridArgs ga;
    const int rc = prepare_grid(env, params, 16, P, scenarios, C, K, integrator, max_steps, tick, stats, violations,
                                &ga.mlp.roll, &ga.pop, &ga.grid);
    if (rc) return rc;
    if (activation != RENV_MLP_TANH && activation != RENV_MLP_RELU) return RENV_E_ARG;
    ga.mlp.params = nullptr;
    ga.mlp.log = LogPtrs<float>{};
    const unsigned blocks = (unsigned)P * ga.pop.ctas;      // <= P C n < 2^31
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    with_activation(activation, [&](auto act) {
        with_flag(ga.mlp.roll.euler, [&](auto euler) {
            cartpole_grid_mlp_kernel<act, euler><<<blocks, kMlpThreads, 0, st>>>(ga);
        });
    });
    return launch_status();
}

// The per-env scenarios of the training entry points (include/renv.h renv_env_scenarios), checked after every check
// of the corresponding plain entry point.
int check_env_scenarios(const renv_env_scenarios *scen, EnvScenPtrs *out)
{
    if (scen == nullptr || scen->rows == nullptr || scen->of_env == nullptr) return RENV_E_NULL;
    if (scen->C < 1 || scen->C > 65535) return RENV_E_SIZE;
    if (!aligned(scen->rows, 16) || !aligned(scen->of_env, 4)) return RENV_E_ALIGN;
    *out = EnvScenPtrs{ scen->rows, scen->of_env, (uint32_t)scen->C };
    return RENV_OK;
}
static_assert(sizeof(renv_alias_entry) == sizeof(uint2) && offsetof(renv_alias_entry, q) == 0 &&
              offsetof(renv_alias_entry, alias) == 4, "alias entry layout differs from MixPtrs::table");
int check_env_scenarios(const renv_env_mixture *mix, MixPtrs *out)
{
    if (mix == nullptr || mix->rows == nullptr || mix->table == nullptr || mix->of_env == nullptr) return RENV_E_NULL;
    if (mix->C < 1 || mix->C > 65535) return RENV_E_SIZE;
    if (!aligned(mix->rows, 16) || !aligned(mix->table, 8) || !aligned(mix->of_env, 4)) return RENV_E_ALIGN;
    *out = MixPtrs{ mix->rows, reinterpret_cast<const uint2 *>(mix->table), mix->of_env, (uint32_t)mix->C };
    return RENV_OK;
}

// The training entry points with per-env rows: per-env scenarios (renv_env_scenarios, the cartpole_scen_* kernels) or
// a scenario mixture (renv_env_mixture, the cartpole_mix_* kernels).  The two forms share every check and launch.
template <bool kMixture> struct RowForm;
template <> struct RowForm<false> {
    using ResetA = ScenResetArgs; using StepA = ScenStepArgs; using RolloutA = ScenRolloutArgs;
    using MlpRolloutA = MlpScenRolloutArgs; using MlpCollectA = MlpScenCollectArgs;
    static auto reset() { return cartpole_scen_reset_kernel; }
    template <bool ln, bool lg> static auto step() { return cartpole_scen_step_kernel<ln, lg>; }
    template <bool e, bool r, bool lg> static auto rollout() { return cartpole_scen_rollout_kernel<e, r, lg>; }
    template <int act, bool e, bool lg> static auto rollout_mlp() { return cartpole_scen_rollout_mlp_kernel<act, e, lg>; }
    template <int act, bool e, bool lg> static auto collect_mlp() { return cartpole_scen_collect_mlp_kernel<act, e, lg>; }
    template <class A> static auto &rows(A &a) { return a.scen; }
};
template <> struct RowForm<true> {
    using ResetA = MixResetArgs; using StepA = MixStepArgs; using RolloutA = MixRolloutArgs;
    using MlpRolloutA = MlpMixRolloutArgs; using MlpCollectA = MlpMixCollectArgs;
    static auto reset() { return cartpole_mix_reset_kernel; }
    template <bool ln, bool lg> static auto step() { return cartpole_mix_step_kernel<ln, lg>; }
    template <bool e, bool r, bool lg> static auto rollout() { return cartpole_mix_rollout_kernel<e, r, lg>; }
    template <int act, bool e, bool lg> static auto rollout_mlp() { return cartpole_mix_rollout_mlp_kernel<act, e, lg>; }
    template <int act, bool e, bool lg> static auto collect_mlp() { return cartpole_mix_collect_mlp_kernel<act, e, lg>; }
    template <class A> static auto &rows(A &a) { return a.mix; }
};

template <class F, class B>
int reset_rows(const renv_cartpole_env *env, const B *scen, const uint8_t *mask, uint64_t tick,
               unsigned long long *violations, void *stream)
{
    typename F::ResetA a;
    int rc = check_env<float>(env, false, &a.reset.env, kNeedEitherElapsed);
    if (rc) return rc;
    if ((rc = to_cfg4<float>(nullptr, &a.reset.dr))) return rc;
    a.reset.mask = mask;
    a.reset.tick = tick;
    a.reset.violations = violations;
    unsigned blocks = 0;
    if ((rc = grid_for(env->n, 256, &blocks))) return rc;
    if ((rc = check_env_scenarios(scen, &F::rows(a)))) return rc;
    F::reset()<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(a);
    return launch_status();
}

// The auto-reset step (renv_cartpole_step_f32 / _lean_f32 / _logged_f32, whichever the env's counter and `log` make
// it) with per-env rows.
template <class F, class B>
int step_rows(const renv_cartpole_env *env, const B *scen, const renv_episode_log *log,
              const uint8_t *action, float *reward, uint8_t *done, uint8_t *truncated, int integrator, int max_steps,
              uint64_t tick, unsigned long long *counters, void *stream)
{
    typename F::StepA sa;
    StepArgs<float> &a = sa.step;
    int rc = check_env<float>(env, false, &a.env, kNeedEitherElapsed);
    if (rc) return rc;
    sa.log = LogPtrs<float>{};
    if (log && (rc = check_log<float>(log, &sa.log))) return rc;
    if (action == nullptr || done == nullptr) return RENV_E_NULL;
    if (!aligned(action, 4) || !aligned(reward, 16) || !aligned(done, 4) || (truncated && !aligned(truncated, 4)))
        return RENV_E_ALIGN;
    if (counters && !aligned(counters, 8)) return RENV_E_ALIGN;
    if (integrator != RENV_EULER && integrator != RENV_SEMI_IMPLICIT) return RENV_E_INTEGRATOR;
    const bool lean = env->elapsed == nullptr;          // the uint16 counter
    if (lean && max_steps > 65535) return RENV_E_SIZE;
    if ((rc = to_cfg4<float>(nullptr, &a.dr))) return rc;
    a.action = action; a.reward = reward; a.done = done; a.truncated = truncated;
    a.euler = integrator == RENV_EULER;
    a.max_steps = max_steps;
    a.tick = tick;
    a.counters = counters;
    unsigned blocks = 0;
    if ((rc = grid_for(env->n, (int64_t)kStepThreads * VecTraits<float>::V, &blocks))) return rc;
    if ((rc = check_env_scenarios(scen, &F::rows(sa)))) return rc;
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    with_flag(lean, [&](auto ln) {
        with_flag(log != nullptr, [&](auto lg) {
            rc = launch_pdl(F::template step<ln, lg>(), blocks, kStepThreads, st, sa);
        });
    });
    return rc;
}

template <class F, class B>
int rollout_rows(const renv_cartpole_env *env, const B *scen, const renv_episode_log *log,
                 const double w[4], double b, int K, int integrator, int max_steps, uint64_t tick, double *stats,
                 unsigned long long *violations, void *stream)
{
    typename F::RolloutA sa;
    int rc = check_env<float>(env, false, &sa.roll.env, kNeedEitherElapsed);
    if (rc) return rc;
    sa.log = LogPtrs<float>{};
    if (log && (rc = check_log<float>(log, &sa.log))) return rc;
    if (stats == nullptr) return RENV_E_NULL;
    const Policy<float> policy = w ? Policy<float>{ (float)w[0], (float)w[1], (float)w[2], (float)w[3], (float)b }
                                   : Policy<float>{ 0.0f, 0.0f, 0.0f, 0.0f, 0.0f };
    if ((rc = check_rollout<float>(stats, K, integrator, max_steps, tick, nullptr, violations, policy, &sa.roll))) return rc;
    if (env->elapsed == nullptr && max_steps > 65535) return RENV_E_SIZE;     // the uint16 counter
    unsigned blocks = 0;
    if ((rc = grid_for(env->n, kRolloutThreads, &blocks))) return rc;
    if ((rc = check_env_scenarios(scen, &F::rows(sa)))) return rc;
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    with_flag(sa.roll.euler, [&](auto euler) {
        with_flag(w == nullptr, [&](auto random) {
            with_flag(log != nullptr, [&](auto lg) {
                F::template rollout<euler, random, lg>()<<<blocks, kRolloutThreads, 0, st>>>(sa);
            });
        });
    });
    return launch_status();
}

template <class F, class B>
int rollout_mlp_rows(const renv_cartpole_env *env, const B *scen, const renv_episode_log *log,
                     const renv_mlp_policy *p, int K, int integrator, int max_steps, uint64_t tick, double *stats,
                     unsigned long long *violations, void *stream)
{
    typename F::MlpRolloutA sa;
    unsigned blocks = 0;
    int rc = prepare_rollout_mlp(env, log, log != nullptr, p, K, integrator, max_steps, tick, nullptr, stats, violations,
                                 &sa.mlp, &blocks);
    if (rc) return rc;
    if ((rc = check_env_scenarios(scen, &F::rows(sa)))) return rc;
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    with_mlp_instance(p->activation, sa.mlp.roll.euler, log != nullptr, [&](auto act, auto euler, auto lg) {
        F::template rollout_mlp<act, euler, lg>()<<<blocks, kMlpThreads, 0, st>>>(sa);
    });
    return launch_status();
}

template <class F, class B>
int collect_mlp_rows(const renv_cartpole_env *env, const B *scen, const renv_episode_log *log,
                     const renv_mlp_policy *p, const renv_trajectory *traj, int sample, int K, int integrator,
                     int max_steps, uint64_t tick, double *stats, unsigned long long *violations, void *stream)
{
    typename F::MlpCollectA sa;
    unsigned blocks = 0;
    int rc = prepare_rollout_mlp(env, log, log != nullptr, p, K, integrator, max_steps, tick, nullptr, stats, violations,
                                 &sa.mlp, &blocks);
    if (rc) return rc;
    if ((rc = check_traj(traj, K, &sa.mlp.traj))) return rc;
    if (sample != 0 && sample != 1) return RENV_E_ARG;
    sa.mlp.sample = sample;
    if ((rc = check_env_scenarios(scen, &F::rows(sa)))) return rc;
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    with_mlp_instance(p->activation, sa.mlp.roll.euler, log != nullptr, [&](auto act, auto euler, auto lg) {
        F::template collect_mlp<act, euler, lg>()<<<blocks, kMlpThreads, 0, st>>>(sa);
    });
    return launch_status();
}

int check_transition_loglik(const renv_transitions *data, int lam, int integrator, const double *xi, int C, int M,
                            const double *eps, double *loglik, double *total, LoglikArgs *a, unsigned *blocks)
{
    if (data == nullptr || data->obs == nullptr || data->next_obs == nullptr || data->action == nullptr ||
        data->window == nullptr || xi == nullptr || eps == nullptr || loglik == nullptr || total == nullptr)
        return RENV_E_NULL;
    if (!aligned(data->obs, 16) || !aligned(data->next_obs, 16) || !aligned(data->window, 4) || !aligned(xi, 16) ||
        !aligned(loglik, 8) || !aligned(total, 8))
        return RENV_E_ALIGN;
    if (data->T < 1 || data->W < 1 || C < 1 || M < 2 || lam < 1 || lam > data->T) return RENV_E_SIZE;
    if (integrator != RENV_EULER && integrator != RENV_SEMI_IMPLICIT) return RENV_E_INTEGRATOR;
    for (int k = 0; k < 4; ++k)
        if (!(eps[k] >= 0.0) || !std::isfinite(eps[k])) return RENV_E_ARG;
    *a = LoglikArgs{ data->obs, data->next_obs, data->action, data->window, xi, loglik, data->T, data->W, C, M, lam,
                     (data->W + kLlWindowsPerCta - 1) / kLlWindowsPerCta, { eps[0], eps[1], eps[2], eps[3] } };
    return grid_for((int64_t)C * a->tiles, 1, blocks);
}

int transition_loglik(const renv_transitions *data, int lam, int integrator, const double *xi, int C, int M,
                      const double *eps, double *loglik, double *total, void *stream)
{
    LoglikArgs a;
    unsigned blocks = 0;
    const int rc = check_transition_loglik(data, lam, integrator, xi, C, M, eps, loglik, total, &a, &blocks);
    if (rc) return rc;
    const cudaStream_t st = static_cast<cudaStream_t>(stream);
    with_flag(integrator == RENV_EULER, [&](auto euler) {
        cartpole_transition_loglik_kernel<euler><<<blocks, kLlThreads, 0, st>>>(a);
    });
    loglik_total_kernel<<<C, kLlSumThreads, 0, st>>>(loglik, data->W, total);
    return launch_status();
}

}  // namespace

extern "C" {

int renv_abi_version(void) { return RENV_ABI_VERSION; }

const char *renv_strerror(int code)
{
    switch (code) {
    case RENV_OK: return "ok";
    case RENV_E_NULL: return "required pointer is NULL";
    case RENV_E_ALIGN: return "pointer or ld violates the alignment contract (16 B data, 4 B byte arrays, ld % V)";
    case RENV_E_SIZE: return "invalid size (n <= 0, ld < n, K <= 0 or grid too large)";
    case RENV_E_DIM: return "dim outside [1, 32] (cart-pole needs 4)";
    case RENV_E_DRTYPE: return "Unknown dr_type";
    case RENV_E_INTEGRATOR: return "unknown integrator";
    case RENV_E_ARG: return "invalid argument";
    default: return code > 0 ? cudaGetErrorString((cudaError_t)code) : "unknown renv status";
    }
}

int renv_dr_sample_f32(float *out, int64_t n, const renv_dr_cfg *cfg, uint64_t seed, uint64_t sample_id0, uint32_t call,
                       unsigned long long *violations, void *stream)
{
    return dr_sample<float>(out, n, cfg, seed, sample_id0, call, violations, stream);
}
int renv_dr_sample_f64(double *out, int64_t n, const renv_dr_cfg *cfg, uint64_t seed, uint64_t sample_id0,
                       uint32_t call, unsigned long long *violations, void *stream)
{
    return dr_sample<double>(out, n, cfg, seed, sample_id0, call, violations, stream);
}

int renv_cartpole_reset_f32(const renv_cartpole_env *env, const uint8_t *mask, uint64_t tick, const renv_dr_cfg *dr,
                            unsigned long long *violations, void *stream)
{
    return cartpole_reset<float>(env, nullptr, mask, tick, dr, violations, stream);
}
int renv_cartpole_reset_f64(const renv_cartpole_env *env, const uint8_t *mask, uint64_t tick, const renv_dr_cfg *dr,
                            unsigned long long *violations, void *stream)
{
    return cartpole_reset<double>(env, nullptr, mask, tick, dr, violations, stream);
}

int renv_cartpole_step_f32(const renv_cartpole_env *env, const uint8_t *action, float *reward, uint8_t *done,
                           uint8_t *truncated, int integrator, int max_steps, int auto_reset, uint64_t tick,
                           const renv_dr_cfg *dr, unsigned long long *counters, void *stream)
{
    return cartpole_step<float, false>(env, nullptr, action, reward, done, truncated, integrator, max_steps, auto_reset,
                                       tick, dr, counters, stream);
}
int renv_cartpole_step_lean_f32(const renv_cartpole_env *env, const uint8_t *action, uint8_t *done, uint8_t *truncated,
                                int integrator, int max_steps, uint64_t tick, const renv_dr_cfg *dr,
                                unsigned long long *counters, void *stream)
{
    return cartpole_step<float, true>(env, nullptr, action, nullptr, done, truncated, integrator, max_steps, 1, tick, dr,
                                      counters, stream);
}
int renv_cartpole_step_f64(const renv_cartpole_env *env, const uint8_t *action, double *reward, uint8_t *done,
                           uint8_t *truncated, int integrator, int max_steps, int auto_reset, uint64_t tick,
                           const renv_dr_cfg *dr, unsigned long long *violations, void *stream)
{
    return cartpole_step<double, false>(env, nullptr, action, reward, done, truncated, integrator, max_steps, auto_reset, tick,
                                 dr, violations, stream);
}

int renv_cartpole_reset_noisy_f32(const renv_cartpole_env *env, const renv_obs_noise *noise, const uint8_t *mask,
                                  uint64_t tick, const renv_dr_cfg *dr, unsigned long long *violations, void *stream)
{
    if (noise == nullptr) return RENV_E_NULL;
    return cartpole_reset<float>(env, noise, mask, tick, dr, violations, stream);
}
int renv_cartpole_reset_noisy_f64(const renv_cartpole_env *env, const renv_obs_noise *noise, const uint8_t *mask,
                                  uint64_t tick, const renv_dr_cfg *dr, unsigned long long *violations, void *stream)
{
    if (noise == nullptr) return RENV_E_NULL;
    return cartpole_reset<double>(env, noise, mask, tick, dr, violations, stream);
}
int renv_cartpole_step_noisy_f32(const renv_cartpole_env *env, const renv_obs_noise *noise, const uint8_t *action,
                                 float *reward, uint8_t *done, uint8_t *truncated, int integrator, int max_steps,
                                 int auto_reset, uint64_t tick, const renv_dr_cfg *dr, unsigned long long *violations,
                                 void *stream)
{
    if (noise == nullptr) return RENV_E_NULL;
    return cartpole_step<float, false>(env, noise, action, reward, done, truncated, integrator, max_steps, auto_reset, tick,
                                dr, violations, stream);
}
int renv_cartpole_step_noisy_f64(const renv_cartpole_env *env, const renv_obs_noise *noise, const uint8_t *action,
                                 double *reward, uint8_t *done, uint8_t *truncated, int integrator, int max_steps,
                                 int auto_reset, uint64_t tick, const renv_dr_cfg *dr, unsigned long long *violations,
                                 void *stream)
{
    if (noise == nullptr) return RENV_E_NULL;
    return cartpole_step<double, false>(env, noise, action, reward, done, truncated, integrator, max_steps, auto_reset, tick,
                                 dr, violations, stream);
}

int renv_cartpole_rollout_f32(const renv_cartpole_env *env, const double w[4], double b, int K, int integrator,
                              int max_steps, uint64_t tick, const renv_dr_cfg *dr, double *stats,
                              unsigned long long *violations, void *stream)
{
    return cartpole_rollout<float>(env, nullptr, w, b, K, integrator, max_steps, tick, dr, stats, violations, stream);
}
int renv_cartpole_rollout_f64(const renv_cartpole_env *env, const double w[4], double b, int K, int integrator,
                              int max_steps, uint64_t tick, const renv_dr_cfg *dr, double *stats,
                              unsigned long long *violations, void *stream)
{
    return cartpole_rollout<double>(env, nullptr, w, b, K, integrator, max_steps, tick, dr, stats, violations, stream);
}

int renv_cartpole_step_logged_f32(const renv_cartpole_env *env, const renv_episode_log *log, const uint8_t *action,
                                  float *reward, uint8_t *done, uint8_t *truncated, int integrator, int max_steps,
                                  uint64_t tick, const renv_dr_cfg *dr, unsigned long long *counters, void *stream)
{
    return cartpole_step<float, false>(env, nullptr, action, reward, done, truncated, integrator, max_steps, 1, tick, dr,
                                       counters, stream, log, true);
}
int renv_cartpole_step_logged_f64(const renv_cartpole_env *env, const renv_episode_log *log, const uint8_t *action,
                                  double *reward, uint8_t *done, uint8_t *truncated, int integrator, int max_steps,
                                  uint64_t tick, const renv_dr_cfg *dr, unsigned long long *counters, void *stream)
{
    return cartpole_step<double, false>(env, nullptr, action, reward, done, truncated, integrator, max_steps, 1, tick, dr,
                                        counters, stream, log, true);
}
int renv_cartpole_rollout_logged_f32(const renv_cartpole_env *env, const renv_episode_log *log, const double w[4], double b,
                                     int K, int integrator, int max_steps, uint64_t tick, const renv_dr_cfg *dr,
                                     double *stats, unsigned long long *violations, void *stream)
{
    return cartpole_rollout<float>(env, nullptr, w, b, K, integrator, max_steps, tick, dr, stats, violations, stream, log,
                                   true);
}
int renv_cartpole_rollout_logged_f64(const renv_cartpole_env *env, const renv_episode_log *log, const double w[4], double b,
                                     int K, int integrator, int max_steps, uint64_t tick, const renv_dr_cfg *dr,
                                     double *stats, unsigned long long *violations, void *stream)
{
    return cartpole_rollout<double>(env, nullptr, w, b, K, integrator, max_steps, tick, dr, stats, violations, stream, log,
                                    true);
}

int renv_cartpole_rollout_noisy_f32(const renv_cartpole_env *env, const renv_obs_noise *noise, const double w[4], double b,
                                    int K, int integrator, int max_steps, uint64_t tick, const renv_dr_cfg *dr,
                                    double *stats, unsigned long long *violations, void *stream)
{
    if (noise == nullptr) return RENV_E_NULL;
    return cartpole_rollout<float>(env, noise, w, b, K, integrator, max_steps, tick, dr, stats, violations, stream);
}
int renv_cartpole_rollout_noisy_f64(const renv_cartpole_env *env, const renv_obs_noise *noise, const double w[4], double b,
                                    int K, int integrator, int max_steps, uint64_t tick, const renv_dr_cfg *dr,
                                    double *stats, unsigned long long *violations, void *stream)
{
    if (noise == nullptr) return RENV_E_NULL;
    return cartpole_rollout<double>(env, noise, w, b, K, integrator, max_steps, tick, dr, stats, violations, stream);
}

int renv_cartpole_policy_actions_mlp_f32(const renv_cartpole_env *env, const renv_mlp_policy *p, uint8_t *action,
                                         float *logits, void *stream)
{
    return policy_mlp(env, p, false, 0, 0, action, nullptr, logits, stream);
}
int renv_cartpole_rollout_mlp_f32(const renv_cartpole_env *env, const renv_mlp_policy *p, int K, int integrator,
                                  int max_steps, uint64_t tick, const renv_dr_cfg *dr, double *stats,
                                  unsigned long long *violations, void *stream)
{
    return rollout_mlp(env, nullptr, false, p, K, integrator, max_steps, tick, dr, stats, violations, stream);
}
int renv_cartpole_rollout_mlp_logged_f32(const renv_cartpole_env *env, const renv_episode_log *log,
                                         const renv_mlp_policy *p, int K, int integrator, int max_steps, uint64_t tick,
                                         const renv_dr_cfg *dr, double *stats, unsigned long long *violations,
                                         void *stream)
{
    return rollout_mlp(env, log, true, p, K, integrator, max_steps, tick, dr, stats, violations, stream);
}
int renv_cartpole_policy_logp_mlp_f32(const renv_cartpole_env *env, const renv_mlp_policy *p, int sample, uint64_t tick,
                                      uint8_t *action, float *logp, float *logits, void *stream)
{
    return policy_mlp(env, p, true, sample, tick, action, logp, logits, stream);
}
int renv_cartpole_collect_mlp_f32(const renv_cartpole_env *env, const renv_mlp_policy *p, const renv_trajectory *traj,
                                  int sample, int K, int integrator, int max_steps, uint64_t tick, const renv_dr_cfg *dr,
                                  double *stats, unsigned long long *violations, void *stream)
{
    return collect_mlp(env, nullptr, false, p, traj, sample, K, integrator, max_steps, tick, dr, stats, violations, stream);
}
int renv_cartpole_collect_mlp_logged_f32(const renv_cartpole_env *env, const renv_episode_log *log,
                                         const renv_mlp_policy *p, const renv_trajectory *traj, int sample, int K,
                                         int integrator, int max_steps, uint64_t tick, const renv_dr_cfg *dr,
                                         double *stats, unsigned long long *violations, void *stream)
{
    return collect_mlp(env, log, true, p, traj, sample, K, integrator, max_steps, tick, dr, stats, violations, stream);
}
int renv_cartpole_gae_mlp_f32(const renv_cartpole_env *env, const renv_mlp_policy *critic, const renv_trajectory *traj,
                              int K, float gamma, float lambda, float *values, float *advantages, float *returns,
                              void *stream)
{
    return gae_mlp(env, critic, traj, K, gamma, lambda, values, advantages, returns, stream);
}

int renv_cartpole_population_linear_f32(const renv_cartpole_env *env, const float *policies, int P, int K,
                                        int integrator, int max_steps, uint64_t tick, const renv_dr_cfg *dr,
                                        double *stats, unsigned long long *violations, void *stream)
{
    return population_linear(env, policies, P, K, integrator, max_steps, tick, dr, stats, violations, stream);
}
int renv_cartpole_population_mlp_f32(const renv_cartpole_env *env, const void *params, int activation, int P, int K,
                                     int integrator, int max_steps, uint64_t tick, const renv_dr_cfg *dr,
                                     double *stats, unsigned long long *violations, void *stream)
{
    return population_mlp(env, params, activation, P, K, integrator, max_steps, tick, dr, stats, violations, stream);
}

int renv_scenario_pack_f32(const renv_dr_cfg *dr, const double task[4], float out[RENV_SCENARIO_FLOATS])
{
    return scenario_pack(dr, task, out);
}
int renv_cartpole_grid_linear_f32(const renv_cartpole_env *env, const float *policies, int P, const float *scenarios,
                                  int C, int K, int integrator, int max_steps, uint64_t tick, double *stats,
                                  unsigned long long *violations, void *stream)
{
    return grid_linear(env, policies, P, scenarios, C, K, integrator, max_steps, tick, stats, violations, stream);
}
int renv_cartpole_grid_mlp_f32(const renv_cartpole_env *env, const void *params, int activation, int P,
                               const float *scenarios, int C, int K, int integrator, int max_steps, uint64_t tick,
                               double *stats, unsigned long long *violations, void *stream)
{
    return grid_mlp(env, params, activation, P, scenarios, C, K, integrator, max_steps, tick, stats, violations, stream);
}

int renv_cartpole_reset_scen_f32(const renv_cartpole_env *env, const renv_env_scenarios *scen, const uint8_t *mask,
                                 uint64_t tick, unsigned long long *violations, void *stream)
{
    return reset_rows<RowForm<false>>(env, scen, mask, tick, violations, stream);
}
int renv_cartpole_step_scen_f32(const renv_cartpole_env *env, const renv_env_scenarios *scen, const renv_episode_log *log,
                                const uint8_t *action, float *reward, uint8_t *done, uint8_t *truncated, int integrator,
                                int max_steps, uint64_t tick, unsigned long long *counters, void *stream)
{
    return step_rows<RowForm<false>>(env, scen, log, action, reward, done, truncated, integrator, max_steps, tick, counters, stream);
}
int renv_cartpole_rollout_scen_f32(const renv_cartpole_env *env, const renv_env_scenarios *scen,
                                   const renv_episode_log *log, const double w[4], double b, int K, int integrator,
                                   int max_steps, uint64_t tick, double *stats, unsigned long long *violations,
                                   void *stream)
{
    return rollout_rows<RowForm<false>>(env, scen, log, w, b, K, integrator, max_steps, tick, stats, violations, stream);
}
int renv_cartpole_rollout_mlp_scen_f32(const renv_cartpole_env *env, const renv_env_scenarios *scen,
                                       const renv_episode_log *log, const renv_mlp_policy *p, int K, int integrator,
                                       int max_steps, uint64_t tick, double *stats, unsigned long long *violations,
                                       void *stream)
{
    return rollout_mlp_rows<RowForm<false>>(env, scen, log, p, K, integrator, max_steps, tick, stats, violations, stream);
}
int renv_cartpole_collect_mlp_scen_f32(const renv_cartpole_env *env, const renv_env_scenarios *scen,
                                       const renv_episode_log *log, const renv_mlp_policy *p, const renv_trajectory *traj,
                                       int sample, int K, int integrator, int max_steps, uint64_t tick, double *stats,
                                       unsigned long long *violations, void *stream)
{
    return collect_mlp_rows<RowForm<false>>(env, scen, log, p, traj, sample, K, integrator, max_steps, tick, stats, violations, stream);
}

int renv_cartpole_reset_mix_f32(const renv_cartpole_env *env, const renv_env_mixture *mix, const uint8_t *mask,
                                uint64_t tick, unsigned long long *violations, void *stream)
{
    return reset_rows<RowForm<true>>(env, mix, mask, tick, violations, stream);
}
int renv_cartpole_step_mix_f32(const renv_cartpole_env *env, const renv_env_mixture *mix, const renv_episode_log *log,
                               const uint8_t *action, float *reward, uint8_t *done, uint8_t *truncated, int integrator,
                               int max_steps, uint64_t tick, unsigned long long *counters, void *stream)
{
    return step_rows<RowForm<true>>(env, mix, log, action, reward, done, truncated, integrator, max_steps, tick, counters,
                                    stream);
}
int renv_cartpole_rollout_mix_f32(const renv_cartpole_env *env, const renv_env_mixture *mix, const renv_episode_log *log,
                                  const double w[4], double b, int K, int integrator, int max_steps, uint64_t tick,
                                  double *stats, unsigned long long *violations, void *stream)
{
    return rollout_rows<RowForm<true>>(env, mix, log, w, b, K, integrator, max_steps, tick, stats, violations, stream);
}
int renv_cartpole_rollout_mlp_mix_f32(const renv_cartpole_env *env, const renv_env_mixture *mix,
                                      const renv_episode_log *log, const renv_mlp_policy *p, int K, int integrator,
                                      int max_steps, uint64_t tick, double *stats, unsigned long long *violations,
                                      void *stream)
{
    return rollout_mlp_rows<RowForm<true>>(env, mix, log, p, K, integrator, max_steps, tick, stats, violations, stream);
}
int renv_cartpole_collect_mlp_mix_f32(const renv_cartpole_env *env, const renv_env_mixture *mix,
                                      const renv_episode_log *log, const renv_mlp_policy *p, const renv_trajectory *traj,
                                      int sample, int K, int integrator, int max_steps, uint64_t tick, double *stats,
                                      unsigned long long *violations, void *stream)
{
    return collect_mlp_rows<RowForm<true>>(env, mix, log, p, traj, sample, K, integrator, max_steps, tick, stats,
                                           violations, stream);
}

int renv_cartpole_transition_loglik_f64(const renv_transitions *data, int lam, int integrator, const double *xi, int C,
                                        int M, const double eps[4], double *loglik, double *total, void *stream)
{
    return transition_loglik(data, lam, integrator, xi, C, M, eps, loglik, total, stream);
}

int renv_cartpole_scalar_serve(renv_scalar_ctrl *ctrl, void *save, uint32_t lease_id, uint64_t lease_ns, void *stream)
{
    if (ctrl == nullptr || save == nullptr) return RENV_E_NULL;
    if (!aligned(ctrl, 64) || !aligned(save, 16)) return RENV_E_ALIGN;
    if (lease_ns == 0 || lease_ns > 1000000000ull) return RENV_E_ARG;      // a lease, not a daemon: at most 1 s idle
    cartpole_scalar_server_kernel<<<1, 32, 0, static_cast<cudaStream_t>(stream)>>>(ctrl, static_cast<ScalarSave *>(save),
                                                                                 lease_id, lease_ns);
    return launch_status();
}

int renv_random_actions_u8(uint8_t *action, int64_t n, uint64_t env_id0, uint64_t seed, uint32_t step, void *stream)
{
    if (action == nullptr) return RENV_E_NULL;
    if (n <= 0) return RENV_E_SIZE;
    if (!aligned(action, 4)) return RENV_E_ALIGN;
    unsigned blocks = 0;
    if (const int rc = grid_for((n + 3) / 4, 256, &blocks)) return rc;
    random_actions_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(action, n, env_id0, seed, step);
    return launch_status();
}

int renv_pack_flags_u8(const uint8_t *flags, uint32_t *bits, int64_t n, void *stream)
{
    if (flags == nullptr || bits == nullptr) return RENV_E_NULL;
    if (n <= 0) return RENV_E_SIZE;
    if (!aligned(flags, 4) || !aligned(bits, 4)) return RENV_E_ALIGN;
    unsigned blocks = 0;
    if (const int rc = grid_for((n + 31) / 32, 256, &blocks)) return rc;
    pack_flags_kernel<<<blocks, 256, 0, static_cast<cudaStream_t>(stream)>>>(flags, bits, n);
    return launch_status();
}

}  // extern "C"
