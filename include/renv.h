/* renv.h -- C ABI of librenv_b200.so: the B200-native RandomCartPole-v0 / DR-sampler hot path.
 *
 * This is the drop-in boundary.  The reference (gabrieletiboni/random-envs) is pure Python and has
 * no FFI; each entry point below names the Python method(s) of the reference it replaces
 * (paths relative to the reference tree).  The shipped binding is ctypes
 * (random_envs_b200/_lib.py); INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - Plain C: pointers, sizes, PODs.  No C++/torch types, no exceptions, no global state.
 *   - Every data pointer is a DEVICE pointer owned by the caller; the library never allocates,
 *     frees or retains memory.  `renv_dr_cfg` / `renv_cartpole_env` are HOST structs read
 *     during the call only.
 *   - Work is enqueued on the caller's `cudaStream_t` (passed as void*); no host sync inside.
 *   - Return value: 0 = OK; < 0 = invalid argument (enum renv_status); > 0 = cudaError_t of the launch.
 *   - Alignment: `state`, `xi`, `reward`, `elapsed`, `out` 16 bytes; `action`, `done`, `truncated`,
 *     `mask` 4 bytes; `ld` a multiple of 4 (f32) or 2 (f64).  Violations return RENV_E_ALIGN.
 *   - Layout: `state` is structure-of-arrays (4, ld): rows x, x_dot, theta, theta_dot.  `xi` is one row per env,
 *     (n, 4) row-major: columns gravity, cart_mass, pole_mass, pole_length (order of
 *     random_envs/random_cartpole.py:104-107,149-155) -- the layout of get_task() / sample_tasks(n), and a reset
 *     rewrites one 32-byte sector instead of four.
 *   - Errors the reference raises from inside the computation are detected on the device and COUNTED in
 *     `counters` (device pointer to RENV_NUM_COUNTERS uint64, caller-zeroed, may be NULL; the entry points that can
 *     only produce the first kind call it `violations`):
 *       counters[0]  gaussian DR dims whose three draws were all < 0.1 (random_env.py:181-186: the reference raises
 *                    Exception('Not all samples were above > 0.1 after 2 attempts'); here the dim is set to 0.1),
 *       counters[1]  step launches x threads that saw an action outside {0, 1} (random_cartpole.py:173-174: the
 *                    reference asserts; here the env is pushed left and the flag is raised).
 *       counters[2]  step CTAs whose tile-ordering wait (renv_cartpole_env.progress) timed out: the progress words
 *                    were not in the state the protocol leaves them in (see there); the step still ran.
 *     The host reads them at its next synchronisation point and raises the reference's exception.
 *   - RNG: counter-based Philox4x32-10, key = seed, counter = (global env id, tick, purpose|slot), purpose 0 initial
 *     state, 1 xi, 2 random action, 3 sample_tasks, 4 observation noise, 5 MLP policy sample, 6 scenario-mixture
 *     row.  `tick` is
 *     the caller's step clock (48 bits used): pass a value that grows by 1 per reset/step call and by K per
 *     K-step rollout (step k of a rollout uses tick + k).  An env starts at most one episode per tick, so
 *     (seed, env_id0 + i, tick) names the episode; results never depend on launch geometry or sharding,
 *     and a K-step rollout at tick t equals K single steps at ticks t .. t+K-1 bit for bit.
 */
#ifndef RENV_B200_H
#define RENV_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define RENV_ABI_VERSION 6
#define RENV_MAX_DIM 32          /* largest task_dim in the suite is 30 (jinja/random_humanoid.py) */
#define RENV_NUM_STATS 6         /* episodes, sum R, sum R^2, min R, max R, sum length */
#define RENV_TILE_ENVS_F32 1024  /* envs per step CTA: the granule of renv_cartpole_env.progress */
#define RENV_TILE_ENVS_F64 512
#define RENV_NUM_COUNTERS 3      /* device-detected error conditions, see `counters` below */

enum renv_status {
    RENV_OK = 0,
    RENV_E_NULL = -1,            /* required pointer is NULL */
    RENV_E_ALIGN = -2,           /* pointer or ld violates the alignment contract */
    RENV_E_SIZE = -3,            /* n <= 0, ld < n, K <= 0 ... */
    RENV_E_DIM = -4,             /* dim outside [1, RENV_MAX_DIM] (or != 4 for cartpole) */
    RENV_E_DRTYPE = -5,          /* unknown dr_type (random_env.py:90 'Unknown dr_type') */
    RENV_E_INTEGRATOR = -6,
    RENV_E_ARG = -7
};

/* random_envs/random_env.py:72-90 -- the string keys of set_dr_distribution. */
enum renv_dr_type {
    RENV_DR_NONE = 0,            /* sampling is None / dr_training False: xi is left alone on reset */
    RENV_DR_UNIFORM = 1,         /* random_env.py:150-151 */
    RENV_DR_TRUNCNORM = 2,       /* random_env.py:153-171 */
    RENV_DR_GAUSSIAN = 3,        /* random_env.py:173-190 */
    RENV_DR_FULLGAUSSIAN = 4     /* random_env.py:192-198 + denormalize_parameters :205-220 */
};

/* random_envs/random_cartpole.py:187-196: 'euler' vs anything else. */
enum renv_integrator { RENV_EULER = 0, RENV_SEMI_IMPLICIT = 1 };

/* Host-side image of RandomEnv's distribution state (random_env.py:102-121 de-interleaved):
 *   uniform:            a = min_task,  b = max_task
 *   truncnorm/gaussian: a = mean_task, b = stdev_task
 *   lb[i] = get_task_lower_bound(i) (used by truncnorm only; gaussian's floor is the literal 0.1).
 *   fullgaussian:       a = mean_task in the normalised [0, 4] space, b / lb = get_task_search_bounds() lo / hi,
 *                       factor = row-major dim x dim matrix F with F F^T = cov_task (e.g. its Cholesky factor):
 *                       xi = denormalize(clip(a + F z, 0, 4)), z ~ N(0, I). */
typedef struct renv_dr_cfg {
    int32_t dr_type;
    int32_t dim;
    double a[RENV_MAX_DIM];
    double b[RENV_MAX_DIM];
    double lb[RENV_MAX_DIM];
    double factor[RENV_MAX_DIM * RENV_MAX_DIM];
} renv_dr_cfg;

/* One shard of cart-pole envs resident in HBM (device pointers, element type T = float | double). */
typedef struct renv_cartpole_env {
    void *state;                 /* T (4, ld)   RandomCartPoleEnv.state            :176,198 */
    void *xi;                    /* T (n, 4)    gravity, cart_mass, pole_mass, pole_length :157-166 */
    int32_t *elapsed;            /* (n) TimeLimit._elapsed_steps (gym 0.21)                 */
    uint32_t *episode;           /* (n) episodes started per env (statistics only; may be NULL)   */
    int32_t *beyond;             /* (n) steps_beyond_done, -1 == None (:207-222); may be NULL when auto_reset */
    uint16_t *elapsed16;         /* (n) the same TimeLimit counter as uint16 (16-byte aligned; fp32 only, max_steps
                                    <= 65535), or NULL.  renv_cartpole_step_lean_f32 steps it; reset zeroes whichever
                                    of elapsed / elapsed16 is set.  `elapsed` may be NULL wherever elapsed16 is set:
                                    in the lean step, reset, the fp32 rollouts (linear, random, MLP, _logged and
                                    _noisy forms), collect and renv_cartpole_step_logged_f32 (then give it
                                    reward = NULL: the lean step's 54 bytes).  These use the int32 counter when
                                    `elapsed` is set, else elapsed16, and return RENV_E_SIZE for max_steps > 65535
                                    with elapsed16 alone.  The population entry points use neither. */
    uint32_t *progress;          /* step-to-step ordering at TILE granularity, or NULL for plain stream order.
                                    2 * ceil(n / RENV_TILE_ENVS_F32 | _F64) uint32, 8-byte aligned, zero-initialised ONCE
                                    by the caller and afterwards touched only by the step entry points: word 2b counts
                                    the step CTAs that have started on tile b, word 2b+1 those that have finished.  A
                                    step CTA runs as soon as ITS tile's previous step has finished instead of waiting
                                    for the whole previous grid, so consecutive step launches of one stream overlap
                                    (also under CUDA-graph replay).  All step launches that share a progress array must
                                    be issued in one stream (or otherwise ordered), as for any in-place update. */
    int64_t n;                   /* envs in this shard */
    int64_t ld;                  /* row stride of state in elements, >= n */
    uint64_t env_id0;            /* global id of env 0 of this shard (rank * n under contiguous sharding) */
    uint64_t seed;               /* Philox key */
} renv_cartpole_env;

/* Episode log of a renv_cartpole_env (device pointers, T as there; row stride = the env's ld).  Every episode of env i
 * that ENDS in a logged step or rollout -- terminated by the thresholds or truncated by the TimeLimit -- writes one
 * record into slot j = count[i] mod capacity, then count[i] += 1: a per-env ring holding the latest
 * min(count[i], capacity) episodes (count[i] - capacity, when positive, were overwritten).  Record slot j of env i is
 * row j * ld + i of each field.  Written by the one thread that resets env i: no atomics, and the content does not
 * depend on launch geometry, tile ordering or sharding; a K-step rollout at tick t logs what K steps at ticks
 * t .. t+K-1 log.  A reset (renv_cartpole_reset_*) abandons running episodes without logging them. */
typedef struct renv_episode_log {
    void *xi;                    /* T (capacity, ld, 4) rows, 16-byte aligned: the task the episode ran under (before the
                                    resample of its reset) */
    void *final_state;           /* T (capacity, ld, 4) rows, 16-byte aligned: x, x_dot, theta, theta_dot after the step
                                    that ended it -- what a step without auto-reset returns (terminal observation) */
    int32_t *length;             /* (capacity, ld), 4-byte aligned: env-steps of the episode, across calls (= its return) */
    uint8_t *truncated;          /* (capacity, ld): 1 when the TimeLimit ended it without meeting the thresholds */
    int64_t *end_tick;           /* (capacity, ld), 8-byte aligned: step clock of the step that ended it */
    int32_t *count;              /* (ld), 4-byte aligned: records written per env since the caller zeroed it */
    int64_t capacity;            /* records per env, 1 <= capacity <= 2^31 - 1 */
} renv_episode_log;

int renv_abi_version(void);
const char *renv_strerror(int code);

/* RandomEnv.sample_tasks(n) -> (n, dim) row-major  (random_env.py:145-203).
 * Sample i uses Philox id = sample_id0 + i and episode field = call.  `violations` (may be NULL) is the
 * RENV_NUM_COUNTERS-element counter array of the Conventions: [0] counts gaussian dims whose three draws were all
 * < 0.1 -- the host raises the reference's Exception('Not all samples were above > 0.1 after 2 attempts') when it
 * is non-zero.
 * dr_type fullgaussian with 17 <= dim <= 32 in fp32 runs its (n x 32) . (32 x 32) contraction on the tensor cores
 * (tcgen05.mma kind::tf32, split into head and tail: fp32-grade products, fp32 accumulation); smaller dims and fp64
 * use FMA chains.  Both draw the same normals; the results agree to 4e-6 of the search-bound width. */
int renv_dr_sample_f32(float *out, int64_t n, const renv_dr_cfg *cfg, uint64_t seed, uint64_t sample_id0,
                       uint32_t call, unsigned long long *violations, void *stream);
int renv_dr_sample_f64(double *out, int64_t n, const renv_dr_cfg *cfg, uint64_t seed, uint64_t sample_id0,
                       uint32_t call, unsigned long long *violations, void *stream);

/* RandomCartPoleEnv.reset (random_cartpole.py:226-229) for every env with mask[i] != 0 (mask NULL = all),
 * preceded by RandomEnv.set_random_task (random_env.py:37-39) when dr != NULL and dr->dr_type != NONE
 * (the README.md:9 / MuJoCo-env behaviour; CartPole's own reset forgets it).  Also zeroes elapsed,
 * sets beyond = -1 and counts the new episode. */
int renv_cartpole_reset_f32(const renv_cartpole_env *env, const uint8_t *mask, uint64_t tick, const renv_dr_cfg *dr,
                            unsigned long long *violations, void *stream);
int renv_cartpole_reset_f64(const renv_cartpole_env *env, const uint8_t *mask, uint64_t tick, const renv_dr_cfg *dr,
                            unsigned long long *violations, void *stream);

/* RandomCartPoleEnv.step (random_cartpole.py:172-224) for all n envs, fused with
 *   TimeLimit.step (gym 0.21; max_steps <= 0 disables)  and
 *   SyncVectorEnv auto-reset (gym 0.21; auto_reset != 0) incl. the DR resample above.
 * action (n) in {0,1}; reward (n) T; done (n) u8; truncated (n) u8 or NULL.
 * With auto_reset the state written back for a finished env is its reset state (the obs gym returns), and
 * `reward` may be NULL: the reward is then 1.0 for every env on every step (:207-212) and is not written.
 * `counters`: RENV_NUM_COUNTERS uint64 (see Conventions). */
int renv_cartpole_step_f32(const renv_cartpole_env *env, const uint8_t *action, float *reward, uint8_t *done,
                           uint8_t *truncated, int integrator, int max_steps, int auto_reset, uint64_t tick,
                           const renv_dr_cfg *dr, unsigned long long *counters, void *stream);
int renv_cartpole_step_f64(const renv_cartpole_env *env, const uint8_t *action, double *reward, uint8_t *done,
                           uint8_t *truncated, int integrator, int max_steps, int auto_reset, uint64_t tick,
                           const renv_dr_cfg *dr, unsigned long long *counters, void *stream);

/* The LEAN auto-reset step: the same env-step with 54 instead of 62 bytes of HBM traffic per env (fp32).  The
 * TimeLimit counter is env->elapsed16 (uint16: max_steps <= 65535) and no reward is written (identically 1.0 under
 * auto-reset, :207-212).  state, xi, done and truncated are bit-identical to renv_cartpole_step_f32 with
 * auto_reset = 1. */
int renv_cartpole_step_lean_f32(const renv_cartpole_env *env, const uint8_t *action, uint8_t *done, uint8_t *truncated,
                                int integrator, int max_steps, uint64_t tick, const renv_dr_cfg *dr,
                                unsigned long long *counters, void *stream);

/* Observation noise of the suite's "Noisy" env variants (jinja/random_hopper.py:28,107-108, random_half_cheetah.py,
 * random_walker2d.py:139-140, random_humanoid.py:193-204): every observation -- after a step and after a reset --
 * is  obs = state + sqrt(noise_level) * N(0, I);  the state itself is not perturbed.  The *_noisy entry points are
 * the plain ones plus this block: `obs` is a DEVICE buffer T (4, ld), 16-byte aligned, that receives the noisy
 * observation (with auto_reset a finished env's row holds the noisy observation of its reset state); `std` =
 * sqrt(noise_level) >= 0.  Normals are Philox draws keyed (seed, env id, tick, purpose 4). */
typedef struct renv_obs_noise {
    void *obs;                   /* T (4, ld) */
    double std;                  /* sqrt(noise_level) */
} renv_obs_noise;

int renv_cartpole_reset_noisy_f32(const renv_cartpole_env *env, const renv_obs_noise *noise, const uint8_t *mask,
                                  uint64_t tick, const renv_dr_cfg *dr, unsigned long long *violations, void *stream);
int renv_cartpole_reset_noisy_f64(const renv_cartpole_env *env, const renv_obs_noise *noise, const uint8_t *mask,
                                  uint64_t tick, const renv_dr_cfg *dr, unsigned long long *violations, void *stream);
int renv_cartpole_step_noisy_f32(const renv_cartpole_env *env, const renv_obs_noise *noise, const uint8_t *action,
                                 float *reward, uint8_t *done, uint8_t *truncated, int integrator, int max_steps,
                                 int auto_reset, uint64_t tick, const renv_dr_cfg *dr, unsigned long long *counters,
                                 void *stream);
int renv_cartpole_step_noisy_f64(const renv_cartpole_env *env, const renv_obs_noise *noise, const uint8_t *action,
                                 double *reward, uint8_t *done, uint8_t *truncated, int integrator, int max_steps,
                                 int auto_reset, uint64_t tick, const renv_dr_cfg *dr, unsigned long long *counters,
                                 void *stream);

/* K fused steps with the linear policy a = [w.s + b > 0] evaluated in-kernel, auto-reset always on.
 * State, xi and counters stay in registers for the K steps (1 <= K <= 2^30).  w == NULL selects the RANDOM policy
 * of the reference's demo loop (test_random_policy.py:26): at tick t env e takes the action bit renv_random_actions_u8
 * would give it for step = t, so the launch equals K x { renv_random_actions_u8; renv_cartpole_step } bit for bit.  stats (device, RENV_NUM_STATS doubles,
 * caller-initialised to {0,0,0,+inf,-inf,0}) is ACCUMULATED with the finished episodes' returns. */
int renv_cartpole_rollout_f32(const renv_cartpole_env *env, const double w[4], double b, int K, int integrator,
                              int max_steps, uint64_t tick, const renv_dr_cfg *dr, double *stats,
                              unsigned long long *violations, void *stream);
int renv_cartpole_rollout_f64(const renv_cartpole_env *env, const double w[4], double b, int K, int integrator,
                              int max_steps, uint64_t tick, const renv_dr_cfg *dr, double *stats,
                              unsigned long long *violations, void *stream);

/* The same with the Noisy variant's observation model: the policy acts on obs = state + std * N(0, I) -- for the
 * first step the content of noise->obs (what the last reset/step left there), afterwards the observation each step
 * or reset would have returned -- and noise->obs is left as K calls of step_noisy would leave it. */
int renv_cartpole_rollout_noisy_f32(const renv_cartpole_env *env, const renv_obs_noise *noise, const double w[4], double b,
                                    int K, int integrator, int max_steps, uint64_t tick, const renv_dr_cfg *dr,
                                    double *stats, unsigned long long *violations, void *stream);
int renv_cartpole_rollout_noisy_f64(const renv_cartpole_env *env, const renv_obs_noise *noise, const double w[4], double b,
                                    int K, int integrator, int max_steps, uint64_t tick, const renv_dr_cfg *dr,
                                    double *stats, unsigned long long *violations, void *stream);

/* renv_cartpole_step_* with auto-reset (implied) and renv_cartpole_rollout_* (w == NULL: random policy), plus the
 * episode log `log` (see renv_episode_log).  State, xi, counters, flags and stats are exactly those of the plain entry
 * points.  log == NULL or a NULL field: RENV_E_NULL; capacity outside [1, 2^31 - 1]: RENV_E_SIZE; misaligned field:
 * RENV_E_ALIGN. */
int renv_cartpole_step_logged_f32(const renv_cartpole_env *env, const renv_episode_log *log, const uint8_t *action,
                                  float *reward, uint8_t *done, uint8_t *truncated, int integrator, int max_steps,
                                  uint64_t tick, const renv_dr_cfg *dr, unsigned long long *counters, void *stream);
int renv_cartpole_step_logged_f64(const renv_cartpole_env *env, const renv_episode_log *log, const uint8_t *action,
                                  double *reward, uint8_t *done, uint8_t *truncated, int integrator, int max_steps,
                                  uint64_t tick, const renv_dr_cfg *dr, unsigned long long *counters, void *stream);
int renv_cartpole_rollout_logged_f32(const renv_cartpole_env *env, const renv_episode_log *log, const double w[4], double b,
                                     int K, int integrator, int max_steps, uint64_t tick, const renv_dr_cfg *dr,
                                     double *stats, unsigned long long *violations, void *stream);
int renv_cartpole_rollout_logged_f64(const renv_cartpole_env *env, const renv_episode_log *log, const double w[4], double b,
                                     int K, int integrator, int max_steps, uint64_t tick, const renv_dr_cfg *dr,
                                     double *stats, unsigned long long *violations, void *stream);

/* A trained MLP policy for the fp32 cart-pole entry points below:
 *     Linear(4, h1) -> act -> Linear(h1, h2) -> act -> Linear(h2, o),  h1, h2 <= 64,  o = 1 or 2,  act = tanh or ReLU,
 * action = argmax(l0, l1), a tie giving 0 (torch.argmax).  `params` is a DEVICE array of RENV_MLP_PARAM_FLOATS fp32,
 * 16-byte aligned, holding the nn.Linear tensors (weight (out, in) row-major, then bias) padded to 64 units:
 *     offset    0  W1 (64, 4)      offset  256  b1 (64)
 *     offset  320  W2 (64, 64)     offset 4416  b2 (64)
 *     offset 4480  W3 (2, 64)      offset 4608  b3 (2)      offset 4610  2 floats of padding (any value)
 * Narrower layers are padded with zero rows / columns / biases (exact: tanh(0) = relu(0) = 0).  A 1-output head
 * Linear(h2, 1) with weight w and bias c is stored as l0 = 0 (zero row 0, b3[0] = 0) and l1 = w.h + c, so that the
 * action is [w.h + c > 0].  The contraction W2 h1 runs on the tensor cores split into TF32 head and tail (3 passes,
 * fp32 accumulation); the logits agree with a float64 evaluation to 1e-5 * max(1, max |logit|). */
#define RENV_MLP_HIDDEN 64
#define RENV_MLP_PARAM_FLOATS 4612
#define RENV_MLP_TANH 0
#define RENV_MLP_RELU 1
typedef struct renv_mlp_policy {
    const void *params;          /* float[RENV_MLP_PARAM_FLOATS], device, 16-byte aligned */
    int32_t activation;          /* RENV_MLP_TANH | RENV_MLP_RELU */
} renv_mlp_policy;

/* The policy's action for each of the env's n envs, from its SoA state: action[i] in {0, 1} (4-byte aligned);
 * `logits` NULL or T (2, ld), 16-byte aligned: row 0 = l0, row 1 = l1.  Errors: NULL env / state / params / action
 * RENV_E_NULL, misaligned RENV_E_ALIGN, unknown activation RENV_E_ARG. */
int renv_cartpole_policy_actions_mlp_f32(const renv_cartpole_env *env, const renv_mlp_policy *p, uint8_t *action,
                                         float *logits, void *stream);
/* renv_cartpole_rollout_f32 with the MLP policy in place of the linear one (the same K range, statistics, counters and
 * argument checks; activation RENV_E_ARG, params as above).  Contract: rollout_mlp(K) at tick t equals K x
 * { renv_cartpole_policy_actions_mlp_f32; renv_cartpole_step_f32 with auto-reset } at ticks t .. t+K-1, bit for bit --
 * state, xi, elapsed, episode counters, stats and (the _logged form, see renv_episode_log) log records. */
int renv_cartpole_rollout_mlp_f32(const renv_cartpole_env *env, const renv_mlp_policy *p, int K, int integrator,
                                  int max_steps, uint64_t tick, const renv_dr_cfg *dr, double *stats,
                                  unsigned long long *violations, void *stream);
int renv_cartpole_rollout_mlp_logged_f32(const renv_cartpole_env *env, const renv_episode_log *log,
                                         const renv_mlp_policy *p, int K, int integrator, int max_steps, uint64_t tick,
                                         const renv_dr_cfg *dr, double *stats, unsigned long long *violations,
                                         void *stream);

/* Stochastic actions of the MLP policy, for on-policy training.  With d = l1 - l0, env e (global id) acting at tick t:
 *   sample = 1:  a = 1 iff u < sigmoid(d), sigmoid in fp32, u = the 24-bit uniform of word x of the Philox block
 *                (seed, e, t, purpose 5, slot 0)  -- a ~ softmax(l0, l1);
 *   sample = 0:  a = argmax(l0, l1), a tie giving 0 (renv_cartpole_policy_actions_mlp_f32's action);
 *   logp = log pi(a | s) = log sigmoid(d) for a = 1, log sigmoid(-d) for a = 0 (in both modes).
 * renv_cartpole_policy_actions_mlp_f32 plus the action rule above at tick `tick` (pass the tick of the step the actions
 * go to): `logp` NULL or float (ld), 4-byte aligned.  Errors as there; `sample` outside {0, 1}: RENV_E_ARG. */
int renv_cartpole_policy_logp_mlp_f32(const renv_cartpole_env *env, const renv_mlp_policy *p, int sample, uint64_t tick,
                                      uint8_t *action, float *logp, float *logits, void *stream);

/* Per-step record of a collected trajectory (device pointers; row stride = the env's ld): step k of env i is row
 * k * ld + i of every field, 0 <= k < K <= capacity. */
typedef struct renv_trajectory {
    float *obs;                  /* (capacity, ld, 4) rows, 16-byte aligned: x, x_dot, theta, theta_dot the action was
                                    chosen from */
    uint8_t *action;             /* (capacity, ld), 4-byte aligned: the action taken */
    uint8_t *done;               /* (capacity, ld), 4-byte aligned: the step ended the episode (terminated or truncated) */
    float *logp;                 /* (capacity, ld), 4-byte aligned, or NULL: log pi(action | obs) */
    uint8_t *truncated;          /* (capacity, ld), 4-byte aligned, or NULL: the TimeLimit ended it (TimeLimit.truncated) */
    float *final_obs;            /* (capacity, ld, 4) rows, 16-byte aligned, or NULL: the state after the step, written
                                    only where done -- the terminal observation auto-reset replaces (the episode log's
                                    final_state); elsewhere left untouched */
    int32_t capacity;            /* steps the buffers hold */
} renv_trajectory;

/* renv_cartpole_rollout_mlp_f32 (_logged: renv_cartpole_rollout_mlp_logged_f32) that also records the trajectory:
 * the reward is 1.0 on every step (:207-212) and is not stored.  Contract: collect(K) at tick t equals K x
 * { record obs = the env's state; renv_cartpole_policy_logp_mlp_f32(sample, tick t + k);
 *   renv_cartpole_step_f32 with auto-reset at tick t + k (done, truncated) }  for k = 0 .. K-1, bit for bit -- every
 * trajectory row, state, xi, elapsed, episode counters, stats and (the _logged form) log records.  With sample = 0 the
 * env, stats and log are exactly those renv_cartpole_rollout_mlp_f32 leaves.  Errors, all before any CUDA call: those of
 * the rollout (K outside [1, 2^30] RENV_E_SIZE, ...); NULL traj / obs / action / done RENV_E_NULL; a misaligned field
 * RENV_E_ALIGN; K > traj->capacity or `sample` outside {0, 1} RENV_E_ARG. */
int renv_cartpole_collect_mlp_f32(const renv_cartpole_env *env, const renv_mlp_policy *p, const renv_trajectory *traj,
                                  int sample, int K, int integrator, int max_steps, uint64_t tick, const renv_dr_cfg *dr,
                                  double *stats, unsigned long long *violations, void *stream);
int renv_cartpole_collect_mlp_logged_f32(const renv_cartpole_env *env, const renv_episode_log *log,
                                         const renv_mlp_policy *p, const renv_trajectory *traj, int sample, int K,
                                         int integrator, int max_steps, uint64_t tick, const renv_dr_cfg *dr,
                                         double *stats, unsigned long long *violations, void *stream);

/* Advantage estimation (GAE) under an MLP critic, for the trajectory renv_cartpole_collect_mlp_f32 has just written.
 * `critic` is a packed 1-output net (l0 = 0): V(s) = l1, the bits renv_cartpole_policy_actions_mlp_f32 returns in logits
 * row 1 for state s.  env->state must be s_K, the state after the collect's last step; only env->state, n and ld are
 * read.  The reward is 1.0 on every step.  For every env i, from k = K-1 down to 0, in fp32 with every operation
 * rounded on its own (no FMA contraction):
 *     v_k   = V(obs[k])
 *     nv_k  = done[k] ? (truncated[k] ? V(final_obs[k]) : 0) : (k + 1 < K ? v_{k+1} : V(s_K))
 *     delta = (1 + gamma * nv_k) - v_k
 *     A_k   = done[k] ? delta : delta + (gamma * lambda) * A_{k+1},   A_K = 0
 *     R_k   = A_k + v_k
 * -- a terminated step bootstraps nothing, a truncated one bootstraps from its terminal observation, and both cut the
 * trace.  final_obs is read only where truncated.  values[k * ld + i] = v_k, advantages[..] = A_k, returns[..] = R_k:
 * (capacity, ld) float arrays, 4-byte aligned.  Errors, all before any CUDA call: NULL env / state / critic / params /
 * traj / obs / done / truncated / final_obs / output RENV_E_NULL; n <= 0, ld < n or K <= 0 RENV_E_SIZE; a misaligned
 * pointer or ld RENV_E_ALIGN; K > traj->capacity, gamma or lambda outside [0, 1] (or NaN), an unknown activation
 * RENV_E_ARG. */
int renv_cartpole_gae_mlp_f32(const renv_cartpole_env *env, const renv_mlp_policy *critic, const renv_trajectory *traj,
                              int K, float gamma, float lambda, float *values, float *advantages, float *returns,
                              void *stream);

/* Population evaluation: P policies, each on the env's E = n envs from a fresh start, with per-member statistics --
 * ES / ARS / CEM over policy weights, population-based training, or the best of several checkpoints under a DR
 * distribution, with common random numbers: member p and member q see the same tasks and initial states.
 * For member p and env j (0 <= j < E), Philox id env_id0 + j for every member:
 *   1. a fresh episode at tick `tick`, exactly as renv_cartpole_reset_f32 (mask NULL) starts one: the initial state
 *      init_state(seed, id, tick); with an active DR config xi is drawn as that reset draws it, otherwise xi is row j of
 *      env->xi;
 *   2. K env-steps at ticks tick + 1 .. tick + K under policy p, with auto-reset, the TimeLimit `max_steps` and the DR
 *      resample on reset, exactly as renv_cartpole_rollout_f32 runs them;
 *   3. the member's finished episodes are ACCUMULATED into stats[p * RENV_NUM_STATS ..] (the rollout's 6 statistics;
 *      the caller initialises each row to {0, 0, 0, +inf, -inf, 0}).
 * Hence stats row p equals, bit for bit, the stats of renv_cartpole_reset_f32 at `tick` followed by
 * renv_cartpole_rollout_f32(policy p, K) at tick + 1 on an env with the same n, seed, env_id0, xi table and DR config:
 * the six values are exact in doubles (integer sums, min, max).  A row depends only on its policy and that
 * configuration, not on P, the member's position or the launch; shards of E with env_id0 offsets combine per member as
 * the rollout's statistics do.  Nothing is written into the env (only env->n, env_id0, seed and, without an active DR
 * config, xi are read); gaussian DR failures are counted into `violations` (may be NULL) as everywhere else.
 * Errors, all before any CUDA call: NULL env / policies / params / stats, or NULL xi when it is read, RENV_E_NULL;
 * P < 1, n <= 0, K outside [1, 2^30] or P * n >= 2^31 RENV_E_SIZE; a misaligned pointer RENV_E_ALIGN (stats 8 bytes,
 * xi 16); an unknown integrator RENV_E_INTEGRATOR; an unknown DR config RENV_E_DRTYPE / RENV_E_DIM.
 *
 * Linear policies: `policies` is P rows of 5 floats w0, w1, w2, w3, b (device, 4-byte aligned); the action is
 * [fma(w3, theta_dot, fma(w2, theta, fma(w1, x_dot, fma(w0, x, b)))) > 0] in fp32 -- the action
 * renv_cartpole_rollout_f32 takes for double w, b that round to these floats. */
int renv_cartpole_population_linear_f32(const renv_cartpole_env *env, const float *policies, int P, int K,
                                        int integrator, int max_steps, uint64_t tick, const renv_dr_cfg *dr,
                                        double *stats, unsigned long long *violations, void *stream);
/* MLP policies: `params` is P rows of RENV_MLP_PARAM_FLOATS floats in the layout of renv_mlp_policy (device; 18,448
 * bytes a row, so every row is 16-byte aligned when the base is), with one `activation` for the whole population
 * (unknown: RENV_E_ARG).  The action is renv_cartpole_rollout_mlp_f32's. */
int renv_cartpole_population_mlp_f32(const renv_cartpole_env *env, const void *params, int activation, int P, int K,
                                     int integrator, int max_steps, uint64_t tick, const renv_dr_cfg *dr,
                                     double *stats, unsigned long long *violations, void *stream);

/* Evaluation grids: P policies x C task scenarios in one launch, with statistics per (policy, scenario) cell -- a
 * return map over the task space, the check of a policy at each boundary of the current ADR ranges, or the choice of a
 * checkpoint over several test distributions.
 *
 * A scenario is a row of RENV_SCENARIO_FLOATS floats (128 bytes, 16-byte aligned in device memory) holding the image of
 * one DR config in the kernels' element type, as renv_scenario_pack_f32 writes it:
 *   float index  0      dr_type (int32 bits): RENV_DR_NONE for a fixed task, else one of the four laws
 *                1      dim (int32 bits, 4)
 *                2..5   a[4]       uniform: lo; truncnorm / gaussian: mean; fullgaussian: mean (normalised space);
 *                                  fixed task: the task (gravity, cart_mass, pole_mass, pole_length)
 *                6..9   b[4]       uniform: float(float(hi) - float(lo)) * 2^-24; truncnorm / gaussian: std;
 *                                  fullgaussian: search-bound lo
 *               10..13  floor[4]   truncnorm: lower bound; gaussian: 0.1; fullgaussian: search-bound hi
 *               14..29  factor[16] fullgaussian: row-major 4 x 4 F with F F^T = cov
 *               30..31  padding (zero) */
#define RENV_SCENARIO_FLOATS 32

/* Host only (no CUDA call, no allocation): scenario row `out` of `dr`, or of the fixed task `task` when `dr` is NULL or
 * RENV_DR_NONE (`task` is not read otherwise).  A distribution row holds exactly the float parameters a launch with
 * that `dr` passes to its kernels, so a grid cell sees the draws a population launch with `dr` sees.  Errors: NULL out,
 * or NULL task for a fixed task, RENV_E_NULL; a non-finite task RENV_E_ARG; an unknown dr_type RENV_E_DRTYPE; dim != 4
 * RENV_E_DIM. */
int renv_scenario_pack_f32(const renv_dr_cfg *dr, const double task[4], float out[RENV_SCENARIO_FLOATS]);

/* With E = env->n: for policy p < P, scenario c < C and env j < E, Philox id env_id0 + j whatever p and c, the cell
 * (p, c) runs what renv_cartpole_population_*_f32 runs for policy row p alone at the same `tick` (a fresh episode at
 * `tick`, then K steps at tick + 1 .. tick + K with auto-reset, the TimeLimit `max_steps` and the resample on reset),
 * with xi taken from scenario row c:
 *   - a row whose dr_type is one of the four laws: as a population launch with `dr` = the config it was packed from;
 *   - any other row (a fixed task): as a population launch with dr = NULL on an xi table whose every row is its task
 *     a[0..3]; the task stays across resets.
 * The cell's finished episodes are ACCUMULATED into stats[(p * C + c) * RENV_NUM_STATS ..] (caller-initialised to
 * {0, 0, 0, +inf, -inf, 0}) and equal, bit for bit, that population launch's row p.  Every cell sees the same initial
 * states and, under one law, the same draws (common random numbers across policies and scenarios); a cell depends on
 * neither P, C nor its position in the grid.  Nothing is written into the env, and only env->n, env_id0 and seed are
 * read (not xi).  Gaussian DR failures are counted into `violations` (may be NULL).
 * Errors, all before any CUDA call: NULL env / policies / params / scenarios / stats RENV_E_NULL; P < 1, C < 1, n <= 0,
 * K outside [1, 2^30] or P * C * n >= 2^31 RENV_E_SIZE; a misaligned pointer RENV_E_ALIGN (scenarios 16 bytes, stats 8,
 * linear policies 4, MLP params 16); an unknown integrator RENV_E_INTEGRATOR; an unknown activation RENV_E_ARG.
 * The policy rows are those of renv_cartpole_population_linear_f32 / renv_cartpole_population_mlp_f32. */
int renv_cartpole_grid_linear_f32(const renv_cartpole_env *env, const float *policies, int P, const float *scenarios,
                                  int C, int K, int integrator, int max_steps, uint64_t tick, double *stats,
                                  unsigned long long *violations, void *stream);
int renv_cartpole_grid_mlp_f32(const renv_cartpole_env *env, const void *params, int activation, int P,
                               const float *scenarios, int C, int K, int integrator, int max_steps, uint64_t tick,
                               double *stats, unsigned long long *violations, void *stream);

/* Per-env task scenarios in the training path: env i has a fixed scenario index of_env[i], and every reset of env i --
 * in reset, in the auto-reset of a step, or inside a rollout or collect -- takes its task from scenario row c = of_env[i]
 * (the rows of the evaluation grids above):
 *   - a row with one of the four laws: xi drawn by the law with Philox (seed, env_id0 + i, tick, purpose 1), exactly as
 *     a launch with the config the row was packed from draws it;
 *   - any other row (a fixed task): xi = the row's a[0..3].
 * So every per-env output of env i -- state, xi, elapsed, episode counters, done / truncated, trajectory rows, logp,
 * episode-log records -- equals, bit for bit, that of a twin env with the same n, seed, env_id0, integrator, TimeLimit
 * and clock whose launches pass the row's law as `dr` (a fixed task: dr = NULL, with the task in every xi row).  Env i
 * depends only on its own row, never on the other envs' assignment or on C.  Several DR distributions (ADR boundary
 * sampling, curricula, mixtures, an empirical task set) thus train in one batch of one launch.
 *
 * The kernels read row min(of_env[i], C - 1), so memory stays in bounds; validating the indices is the caller's job.
 * Rollout and collect accumulate the finished episodes of the envs of scenario c into stats[c * RENV_NUM_STATS ..], a
 * (C, RENV_NUM_STATS) array initialised like the plain stats; each row is exact in doubles (integer sums, a min and a
 * max), whatever the order of the atomics.  fp32 only; `log` may be NULL, otherwise it is checked and written as by the
 * _logged forms.  Errors, all before any CUDA call: every check of the corresponding plain entry point with its code,
 * then NULL scen, rows or of_env RENV_E_NULL; C outside [1, 65535] RENV_E_SIZE; misaligned rows or of_env
 * RENV_E_ALIGN. */
typedef struct renv_env_scenarios {
    const float *rows;        /* (C, RENV_SCENARIO_FLOATS) device rows, 16-byte aligned, as renv_scenario_pack_f32 writes them */
    const uint16_t *of_env;   /* (n) device, 4-byte aligned: the scenario of env i, < C */
    int32_t C;                /* 1 <= C <= 65535 */
} renv_env_scenarios;

/* renv_cartpole_reset_f32 with env i's row in place of `dr`. */
int renv_cartpole_reset_scen_f32(const renv_cartpole_env *env, const renv_env_scenarios *scen, const uint8_t *mask,
                                 uint64_t tick, unsigned long long *violations, void *stream);
/* The auto-reset step: the int32 TimeLimit counter when env->elapsed is set, else the uint16 one (max_steps <= 65535);
 * reward == NULL drops the reward store (with the uint16 counter: the 54-byte step of renv_cartpole_step_lean_f32).
 * With `log`, the step of renv_cartpole_step_logged_f32.  Only the CTA reset pass reads of_env and the rows. */
int renv_cartpole_step_scen_f32(const renv_cartpole_env *env, const renv_env_scenarios *scen, const renv_episode_log *log,
                                const uint8_t *action, float *reward, uint8_t *done, uint8_t *truncated, int integrator,
                                int max_steps, uint64_t tick, unsigned long long *counters, void *stream);
/* renv_cartpole_rollout_f32 (linear policy, or the random policy with w == NULL), statistics per scenario. */
int renv_cartpole_rollout_scen_f32(const renv_cartpole_env *env, const renv_env_scenarios *scen,
                                   const renv_episode_log *log, const double w[4], double b, int K, int integrator,
                                   int max_steps, uint64_t tick, double *stats, unsigned long long *violations,
                                   void *stream);
/* renv_cartpole_rollout_mlp_f32, statistics per scenario. */
int renv_cartpole_rollout_mlp_scen_f32(const renv_cartpole_env *env, const renv_env_scenarios *scen,
                                       const renv_episode_log *log, const renv_mlp_policy *p, int K, int integrator,
                                       int max_steps, uint64_t tick, double *stats, unsigned long long *violations,
                                       void *stream);
/* renv_cartpole_collect_mlp_f32, statistics per scenario. */
int renv_cartpole_collect_mlp_scen_f32(const renv_cartpole_env *env, const renv_env_scenarios *scen,
                                       const renv_episode_log *log, const renv_mlp_policy *p, const renv_trajectory *traj,
                                       int sample, int K, int integrator, int max_steps, uint64_t tick, double *stats,
                                       unsigned long long *violations, void *stream);

/* Scenario mixtures in the training path: every reset of env i -- in reset, in the auto-reset of a step, or inside a
 * rollout or collect -- at clock tick t draws its scenario row c from a C-entry alias table:
 *   (x, y) = words 0 and 1 of the Philox block (seed, env_id0 + i, t, purpose 6, slot 0);
 *   j = (uint64_t)x * C >> 32;   c = y < table[j].q ? j : table[j].alias.
 * Row c is P(c) = sum over j of [j == c] (q_j / 2^32) / C + [alias_j == c] (1 - q_j / 2^32) / C, an integer count over
 * 2^64.  The reset is then exactly the per-env scenario reset above with row c (a law row draws xi with purpose 1 at
 * (env_id0 + i, t), a fixed row gives its task), and of_env[i] = c is stored.  So every per-env output of env i equals,
 * bit for bit, that of a renv_env_scenarios twin whose of_env[i] is set to the drawn row before each reset.
 *
 * of_env[i] holds the row of env i's running episode; the kernels write it.  C marks an episode that began before the
 * mixture was installed.  Rollout and collect accumulate each finished episode into stats[min(of_env, C) *
 * RENV_NUM_STATS ..] of the reset that began it: a (C + 1, RENV_NUM_STATS) array, initialised like the plain stats,
 * whose row C holds the episodes that began before the mixture.  Each row is exact in doubles.  A bad alias is clamped
 * to C - 1; building the table is the caller's job.  fp32 only; `log` may be NULL or an episode log.  Errors, all before
 * any CUDA call: every check of the corresponding plain entry point with its code, then NULL mix, rows, table or of_env
 * RENV_E_NULL; C outside [1, 65535] RENV_E_SIZE; misaligned rows, table or of_env RENV_E_ALIGN. */
typedef struct renv_alias_entry {
    uint32_t q;               /* column j keeps row j when y < q */
    uint16_t alias;           /* ... and gives row alias otherwise */
    uint16_t pad;
} renv_alias_entry;

typedef struct renv_env_mixture {
    const float *rows;                /* (C, RENV_SCENARIO_FLOATS) device rows, 16-byte aligned */
    const renv_alias_entry *table;    /* (C) device, 8-byte aligned */
    uint16_t *of_env;                 /* (n) device, 4-byte aligned: the row of env i's running episode (written) */
    int32_t C;                        /* 1 <= C <= 65535 */
} renv_env_mixture;

/* renv_cartpole_reset_scen_f32 with the drawn row. */
int renv_cartpole_reset_mix_f32(const renv_cartpole_env *env, const renv_env_mixture *mix, const uint8_t *mask,
                                uint64_t tick, unsigned long long *violations, void *stream);
/* renv_cartpole_step_scen_f32 with the drawn row: only the CTA reset pass draws and reads the table and rows. */
int renv_cartpole_step_mix_f32(const renv_cartpole_env *env, const renv_env_mixture *mix, const renv_episode_log *log,
                               const uint8_t *action, float *reward, uint8_t *done, uint8_t *truncated, int integrator,
                               int max_steps, uint64_t tick, unsigned long long *counters, void *stream);
/* renv_cartpole_rollout_scen_f32 with the drawn rows, statistics per row into (C + 1, RENV_NUM_STATS). */
int renv_cartpole_rollout_mix_f32(const renv_cartpole_env *env, const renv_env_mixture *mix, const renv_episode_log *log,
                                  const double w[4], double b, int K, int integrator, int max_steps, uint64_t tick,
                                  double *stats, unsigned long long *violations, void *stream);
/* renv_cartpole_rollout_mlp_scen_f32 with the drawn rows. */
int renv_cartpole_rollout_mlp_mix_f32(const renv_cartpole_env *env, const renv_env_mixture *mix,
                                      const renv_episode_log *log, const renv_mlp_policy *p, int K, int integrator,
                                      int max_steps, uint64_t tick, double *stats, unsigned long long *violations,
                                      void *stream);
/* renv_cartpole_collect_mlp_scen_f32 with the drawn rows. */
int renv_cartpole_collect_mlp_mix_f32(const renv_cartpole_env *env, const renv_env_mixture *mix,
                                      const renv_episode_log *log, const renv_mlp_policy *p, const renv_trajectory *traj,
                                      int sample, int K, int integrator, int max_steps, uint64_t tick, double *stats,
                                      unsigned long long *violations, void *stream);

/* Recorded cart-pole transitions for offline DR fitting (device pointers): transition i is (obs[i], action[i],
 * next_obs[i]), and `window` lists the W start indices t that are scored (t + lam <= T; windows crossing an episode
 * boundary are the caller's to leave out). */
typedef struct renv_transitions {
    const double *obs;           /* (T, 4) rows x, x_dot, theta, theta_dot, 16-byte aligned */
    const double *next_obs;      /* (T, 4) rows, 16-byte aligned: the observation after action[i] */
    const uint8_t *action;       /* (T) in {0, 1} */
    const int32_t *window;       /* (W) start indices, 4-byte aligned */
    int64_t T;
    int32_t W;
} renv_transitions;

/* Log-likelihood of C candidate task distributions on recorded transitions, the objective DROPO-style offline DR
 * fitting maximises (it replaces set_task / state assignment / step, random_cartpole.py:157-166,172-205, called once per
 * candidate, transition, sample and step).  Candidate c is given by M >= 2 task samples xi (C, M, 4) rows, 16-byte
 * aligned (gravity, cart_mass, pole_mass, pole_length).  For window w with start t and sample m:
 *     s_m = lam applications of RandomCartPoleEnv's dynamics (:176-196, the fp64 parity arithmetic of step; termination
 *           is ignored: no TimeLimit, no reset) under xi[c, m] and actions action[t .. t+lam-1], from obs[t]
 *     y = next_obs[t+lam-1],  mu = mean_m s_m,  Sigma = 1/(M-1) sum_m (s_m - mu)(s_m - mu)' (numpy cov, ddof 1)
 *     S = Sigma + diag(eps)
 *     loglik[c * W + w] = -1/2 (y - mu)' S^-1 (y - mu) - 1/2 log det S - 2 log(2 pi)
 *                         (= scipy.stats.multivariate_normal.logpdf(y, mu, S));
 *                         -inf when the Cholesky factorisation of S meets a pivot <= 0 or NaN;
 *                         NaN when t < 0 or t + lam > T (a device-side guard; validate windows on the host)
 *     total[c] = sum_w loglik[c, w]  (fixed order, compensated: within a few ulp of the exact sum of the values)
 * eps (4 doubles, host) >= 0, per dimension: under Euler with lam = 1 the rows x and theta of s_m do not depend on xi,
 * so two rows of Sigma are exactly zero and S is singular without it; with observation noise of std sigma in obs and
 * next_obs, eps = 2 sigma^2 is the natural floor.  loglik (C, W) and total (C) are device doubles, 8-byte aligned.
 * Bitwise reproducible: loglik[c, .] and total[c] depend only on (data, windows, xi[c], eps, lam, integrator), not on C,
 * the other candidates or the launch, and two identical calls give identical bits.  Errors, all before any CUDA call:
 * NULL data / pointer RENV_E_NULL; a misaligned pointer RENV_E_ALIGN; T, W, C < 1, M < 2, lam < 1 or lam > T
 * RENV_E_SIZE; an unknown integrator RENV_E_INTEGRATOR; eps < 0 or not finite RENV_E_ARG. */
int renv_cartpole_transition_loglik_f64(const renv_transitions *data, int lam, int integrator, const double *xi, int C,
                                        int M, const double eps[4], double *loglik, double *total, void *stream);

/* The SCALAR drop-in env (gym.make('RandomCartPole-v0'): RandomCartPoleEnv.step / reset, random_cartpole.py:172-229,
 * one env, one host call per step) served by a resident one-warp kernel instead of one launch + synchronise per call.
 * `ctrl` is PINNED, DEVICE-MAPPED HOST memory (zero-initialised once): the host rings a request in by writing
 * `request = (seq << 8) | op` (seq grows by 1 per request, 24 bits; op 0 / 1 = step(action); 2 = reset, 3 = set state,
 * 4 = set xi, 5 = configure, 6 = exit, each reading the `arg` / `arg_u64` fields that the host wrote BEFORE the request
 * word -- see csrc/renv_scalar_server.cuh for the field meanings) and spins on `ack == seq`; the results are in
 * state / obs / xi / reward / done / beyond / violations (or, for a step, already in `next[action]`, see below).  `save` is RENV_SCALAR_SAVE_BYTES of zero-initialised DEVICE
 * memory that carries the env between kernel instances: the kernel is a lease -- after `lease_ns` without a request it
 * stores its registers there, sets ctrl->exited = lease_id and exits; the caller launches the next instance (lease_id
 * + 1) when it has a request and sees exited == the id it launched last.  One instance at a time per ctrl block. */
#define RENV_SCALAR_SAVE_BYTES 512
typedef struct renv_scalar_ctrl {
    uint32_t request;            /* host -> device */
    uint32_t pad0[15];
    double arg[16];              /* host -> device: arguments of ops >= 2 */
    uint64_t arg_u64[8];
    double state[4];             /* device -> host: x, x_dot, theta, theta_dot after the request */
    double obs[4];               /*   Noisy variant: state + sqrt(noise_level) N(0, I) */
    double xi[4];                /*   gravity, cart_mass, pole_mass, pole_length (written by ops >= 2) */
    double reward;
    int32_t done;
    int32_t beyond;              /*   steps_beyond_done, -1 == None */
    uint32_t violations;         /*   gaussian DR dims that failed three times (reset with resample) */
    uint32_t pad1;
    uint32_t ack;                /* device -> host: seq of the last request served */
    uint32_t exited;             /* device -> host: lease id of the instance that has exited */
    uint32_t pad2[16];
    /* Look-ahead (device -> host; enabled by arg_u64[5] != 0 of a configure request): after serving request `next_seq`
     * the kernel also publishes what step(0) and step(1) would return from the state it is in now.  A host that finds
     * next_seq == the seq of its last request takes next[action] as the result of its next step AT ONCE and rings that
     * step in as op 8 + action WITHOUT waiting (ops 8 / 9 are not acknowledged and write no result block; at most one
     * request is outstanding: before it rings again the host waits for next_seq == that step's seq), which takes the
     * PCIe round trip off the step's critical path.  The kernel counts the step clock itself for the Noisy variant's
     * observations (tick of the last reset + 1 per step, or arg_u64[4] of a configure request). */
    struct renv_scalar_outcome {
        double state[4];
        double obs[4];           /*   Noisy variant */
        double reward;
        int32_t done;
        int32_t beyond;
        uint32_t pad[12];
    } next[2];
    uint32_t next_seq;           /* release-stored after next[0..1] */
    uint32_t pad3[15];
} renv_scalar_ctrl;
int renv_cartpole_scalar_serve(renv_scalar_ctrl *ctrl, void *save, uint32_t lease_id, uint64_t lease_ns, void *stream);

/* action_space.sample() for n envs (test_random_policy.py:26): env e at clock `step` takes bit (step & 127) of its own
 * Philox block (e, step >> 7), purpose 2 -- one block holds an env's Bernoulli(1/2) actions for 128 consecutive steps. */
int renv_random_actions_u8(uint8_t *action, int64_t n, uint64_t env_id0, uint64_t seed, uint32_t step,
                           void *stream);

/* Host-path helper (no counterpart in the reference, whose envs live in host memory): packs n byte flags (0 / non-zero,
 * the `done` / `truncated` vectors of renv_cartpole_step_*) into bits -- bit (i & 7) of byte i >> 3, numpy's
 * bitorder "little" -- so that they cross PCIe as n / 8 bytes.  `bits` holds ceil(n / 32) 32-bit words; both pointers
 * 4-byte aligned (16-byte aligned flags take the vector path). */
int renv_pack_flags_u8(const uint8_t *flags, uint32_t *bits, int64_t n, void *stream);

#ifdef __cplusplus
}
#endif
#endif /* RENV_B200_H */
