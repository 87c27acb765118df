"""Vectorised, tensor-in/tensor-out RandomCartPole: N envs resident in HBM, one kernel per call.

Same method names as the reference's single env (random_cartpole.py / random_env.py): ``reset``,
``step``, ``seed``, ``get_task``, ``set_task``, ``set_random_task``, ``set_dr_distribution``,
``set_dr_training`` ...; arguments and results are batched torch CUDA tensors:

    reset()        -> obs (N, 4)
    step(actions)  -> obs (N, 4), reward (N,), done (N,) bool, info {'TimeLimit.truncated': (N,) bool}
    get_task()     -> (N, 4)            set_task(Tensor(N, 4) | g, m_c, m_p, l)
    rollout(w, b, K) -> None            (K fused steps of the linear policy a = [w.s + b > 0] or of an MLPPolicy)
    evaluate_population(policies, K) -> (P, 6)   (P policies on common tasks from fresh starts; the env is untouched)
    evaluate_grid(policies, scenarios, K) -> (P, C, 6)   (the same for each of C task scenarios, in one kernel)
    set_scenarios(scenarios, assignment)  (env i resets from scenario assignment[i] in reset / step / rollout / collect)
    set_scenario_mixture(scenarios, weights)  (every reset draws its scenario from the weighted rows, on the device)
    set_mixture_weights(weights)        (new weights for the next resets; rows, running episodes and statistics kept)
    scenario_stats() -> (C, 6)          (returns of the episodes finished inside rollouts, per scenario)
    policy_actions(policy) -> (N,)      (the MLPPolicy's actions for the current observations, ready for step)
    collect(policy, K) -> Trajectory    (K fused steps under the sampled policy, every step recorded for training)
    gae(traj, critic) -> Trajectory     (values, GAE advantages and returns of that trajectory under an MLP critic)
    episode_stats()  -> dict            (returns of the episodes finished inside rollouts)
    start_episode_log(R) -> EpisodeLog  (per-env record of every episode that ends in step / rollout)

``step`` fuses what the reference stack does in three Python layers: ``RandomCartPoleEnv.step``
(random_cartpole.py:172-224), gym 0.21 ``TimeLimit.step`` (max_episode_steps=500, :294) and gym 0.21
``SyncVectorEnv`` auto-reset, including the DR resample on reset when ``dr_training`` is on
(README.md:9; random_env.py:37-39).  The returned tensors are views of the env's own buffers (the
reference's ``obs`` likewise aliases ``state``): they are overwritten by the next call.

State is stored structure-of-arrays ``(4, ld)`` so that the kernels read and write 128-bit coalesced
vectors (``obs`` is the transposed ``(N, 4)`` view); xi is stored one row per env, ``(N, 4)``, which is
what ``get_task`` returns.
"""
import ctypes
import math

import numpy as np

from . import _device, _lib
from .episode_log import EpisodeLog
from .mlp_policy import PARAM_FLOATS, MLPPolicy, MLPPopulation
from .random_env import RandomEnv
from .trajectory import Trajectory
from .xi_tables import get_table

_TABLE = get_table("RandomCartPole-v0")
NOMINAL_TASK = (9.8, 1.0, 0.1, 0.5)                 # random_cartpole.py:74-78
THETA_THRESHOLD_RADIANS = 12 * 2 * math.pi / 360   # :85
X_THRESHOLD = 2.4                                  # :86
MAX_EPISODE_STEPS = 500                            # :294
# entry points that end episodes: a _logged variant (taking the log after env) runs them while a log is attached
_LOGGED_ENTRIES = ("step", "step_lean", "rollout", "rollout_mlp", "collect_mlp")
_NOISY_ENTRIES = ("reset", "step", "rollout")       # a _noisy variant takes the obs-noise block after env


_EMPTY_STATS = [0.0, 0.0, 0.0, math.inf, -math.inf, 0.0]


def _combine_stats(rows):
    """(R, 6) statistics rows -> their 6-vector combination (sum, sum, sum, min, max, sum), on their device.  Exact:
    the sums are of integers below 2^53."""
    t = _device.torch()
    return t.stack([rows[:, 0].sum(), rows[:, 1].sum(), rows[:, 2].sum(), rows[:, 3].min(), rows[:, 4].max(),
                    rows[:, 5].sum()])


def _mixture_table(weights, C):
    """(weights as a float64 numpy array, the (C,) int64 alias table of include/renv.h renv_env_mixture) of C mixture
    weights; raises ValueError on bad weights.  Vose's method in float64, then q rounded to an integer over 2^32; two
    rules hold exactly: a weight-0 row is never drawn (its q is 0 and no column aliases it), and a column that keeps
    all its mass aliases itself (so y < q failing at y = 2^32 - 1 still draws it).  Entry j is q | alias << 32."""
    t = _device.torch()
    if isinstance(weights, t.Tensor):
        weights = weights.detach().to("cpu", t.float64).numpy()        # the one synchronisation of a device tensor
    w = np.array(weights, dtype=np.float64)
    if w.shape != (C,):
        raise ValueError("the mixture weights must have shape (%d,), got %s" % (C, w.shape))
    if not np.all(np.isfinite(w)) or np.any(w < 0):
        raise ValueError("the mixture weights must be finite and >= 0")
    total = w.sum()
    if not total > 0:
        raise ValueError("the mixture weights must have a positive sum")
    p = w * (C / total)
    q = np.ones(C, dtype=np.float64)
    alias = np.arange(C, dtype=np.int64)
    small = [j for j in range(C) if p[j] < 1.0]
    large = [j for j in range(C) if p[j] >= 1.0]
    while small and large:
        s, l = small.pop(), large.pop()
        q[s], alias[s] = p[s], l
        p[l] -= 1.0 - p[s]
        (small if p[l] < 1.0 else large).append(l)
    # left over by rounding: columns whose mass is (nearly) 1 keep it, except a weight-0 row, which gives it away
    heaviest = int(np.argmax(w))
    for j in small + large:
        q[j], alias[j] = (1.0, j) if w[j] > 0 else (0.0, heaviest)
    qi = np.minimum(np.rint(q * 2.0 ** 32), 2.0 ** 32).astype(np.int64)
    qi[w == 0] = 0
    keep = qi >= 2 ** 32
    alias[keep] = np.nonzero(keep)[0]
    qi[keep] = 2 ** 32 - 1
    return w, qi | (alias << 32)


def _round_up(x, m):
    return (x + m - 1) // m * m


class RandomCartPoleVecEnv(RandomEnv):
    """N domain-randomised cart-poles stepped by hand-written sm_100a kernels."""

    def __init__(self, num_envs, dtype="float32", device=None, seed=0, env_id0=0,
                 max_episode_steps=MAX_EPISODE_STEPS, auto_reset=True, kinematics_integrator="euler",
                 track_truncated=True, validate_actions=True, track_episodes=True, noisy=False, noise_level=1e-4,
                 lean=False, tile_ordering="auto", pack_host_flags=True, _int32_counter=False):
        RandomEnv.__init__(self)
        if num_envs <= 0:
            raise ValueError("num_envs must be positive")
        self.num_envs = int(num_envs)
        # step_host_*: done / truncated cross PCIe as bits (renv_pack_flags_u8) and are unpacked on the host
        self.pack_host_flags = bool(pack_host_flags)
        self._dtype_name = str(dtype).replace("torch.", "")
        if self._dtype_name not in ("float32", "float64"):
            raise ValueError("dtype must be float32 or float64")
        self._device_arg = device
        self._seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        self.env_id0 = int(env_id0)
        self.max_episode_steps = 0 if max_episode_steps is None else int(max_episode_steps)
        self.auto_reset = bool(auto_reset)
        self.kinematics_integrator = kinematics_integrator
        self.track_truncated = bool(track_truncated)
        self.validate_actions = bool(validate_actions)
        self.track_episodes = bool(track_episodes)
        # the suite's "Noisy" variants (jinja/random_hopper.py:16,28,107-108): obs = state + sqrt(noise_level) * N(0, I)
        self.noisy = bool(noisy)
        self.noise_level = float(noise_level)
        if self.noise_level < 0:
            raise ValueError("noise_level must be >= 0")
        # lean step (include/renv.h renv_cartpole_step_lean_f32): uint16 TimeLimit counter, no reward store -- 54 instead
        # of 62 bytes of HBM traffic per env-step; state / done / truncated bit-identical.  The default env takes the
        # same step whenever it can (see _counter16_fits); lean=True only insists on it, and keeps rollout(), collect()
        # and the episode log refused as they were before the default took that step.
        self.lean = bool(lean)
        self._int32_counter = bool(_int32_counter) and not self.lean     # tests: the int32 layout whatever the settings
        if self.lean and (self._dtype_name != "float32" or not self.auto_reset or self.noisy
                          or not 0 < self.max_episode_steps <= 65535):
            raise ValueError("lean=True needs float32, auto_reset, no observation noise and 0 < max_episode_steps <= 65535")

        # step-to-step ordering per 1024-env tile instead of per launch (include/renv.h renv_cartpole_env.progress):
        # consecutive step() launches of one stream overlap; False = plain stream order between launches.  "auto": on
        # up to 2^21 envs, where the launch-to-launch bubble is >= 10 % of a step; beyond that (and for steps issued
        # from several streams / parallel graph branches) the per-CTA ticket round trip costs more than it saves
        self.tile_ordering = (self.num_envs <= (1 << 21)) if tile_ordering == "auto" else bool(tile_ordering)

        self.dyn_ind_to_name = dict(enumerate(_TABLE.names))
        self.original_task = np.array(NOMINAL_TASK)
        self.task_dim = 4
        self.min_task = np.zeros(4)
        self.max_task = np.zeros(4)
        self.mean_task = np.zeros(4)
        self.stdev_task = np.zeros(4)
        self.reward_threshold = _TABLE.reward_threshold
        self.theta_threshold_radians = THETA_THRESHOLD_RADIANS
        self.x_threshold = X_THRESHOLD
        self.force_mag, self.tau = 10.0, 0.02
        self.polemass_length = 0.05     # frozen, as in the reference (:79 vs :157-166)
        self._buffers = None
        self._episode_log = None        # EpisodeLog attached by start_episode_log
        self._scen = None               # per-env scenarios (set_scenarios) or a mixture (set_scenario_mixture): rows,
                                        # of_env, stats, the C struct; a mixture also its weights and alias table
        self._scen_version = 0          # bumped whenever _scen changes (the step plan holds a pointer to its struct)
        self._cfg_cache = None
        self._cfg_key = None
        self._tick = 0                  # step clock: Philox episode key; +1 per reset/step, +K per rollout
        self.seed_dr(self._seed)        # set_random_task / sample_tasks draw from the constructor seed's stream

    # ---- xi tables (random_cartpole.py:123-147) ----------------------------------------------------
    def get_search_bounds_mean(self, index):
        return _TABLE.search_bounds[index]

    def get_task_lower_bound(self, index):
        return _TABLE.lower_bounds[index]

    # ---- buffers ----------------------------------------------------------------------------------
    def _counter16_fits(self):
        """The env's settings allow the uint16 TimeLimit counter: float32, auto-reset, no observation noise and
        0 < max_episode_steps <= 65535.  Then the counter never exceeds 65535 and the reward is 1.0 on every step, so
        ``step`` moves 54 instead of 62 bytes per env (no reward store) with bit-identical results."""
        return self._dtype_name == "float32" and self.auto_reset and not self.noisy \
            and 0 < self.max_episode_steps <= 65535

    def _check_counter(self):
        """Widen the uint16 counter to int32 once a setting changed since allocation rules it out (auto_reset,
        noisy and max_episode_steps are plain attributes).  One-way: a widened counter may have counted past 65535."""
        b = self._buffers
        if b["elapsed16"] is not None and not self.lean and not self._counter16_fits():
            t = _device.torch()
            b["elapsed"] = b["elapsed16"].to(t.int32) & 0xFFFF
            b["elapsed16"] = None
            self._refresh_env_struct()

    @property
    def torch_dtype(self):
        t = _device.torch()
        return t.float32 if self._dtype_name == "float32" else t.float64

    @property
    def device(self):
        return self._alloc()["device"]

    def _alloc(self):
        if self._buffers is not None:
            return self._buffers
        t = _device.torch()
        dev = _device.require_cuda(self._device_arg)
        _lib.load()
        n, ld = self.num_envs, _round_up(self.num_envs, 32)
        dt = self.torch_dtype
        b = dict(device=dev, ld=ld)
        b["state"] = t.zeros((4, ld), dtype=dt, device=dev)
        b["xi"] = t.tensor(NOMINAL_TASK, dtype=dt, device=dev).reshape(1, 4).repeat(ld, 1).contiguous()   # (ld, 4) rows
        counter16 = self.lean or (self._counter16_fits() and not self._int32_counter)
        b["elapsed16"] = t.zeros(ld, dtype=t.int16, device=dev) if counter16 else None     # uint16 bit pattern
        b["elapsed"] = b["elapsed16"] if counter16 else t.zeros(ld, dtype=t.int32, device=dev)  # the counter, either layout
        b["episode"] = t.zeros(ld, dtype=t.int32, device=dev)       # uint32 bit pattern
        b["beyond"] = t.full((ld,), -1, dtype=t.int32, device=dev)
        b["reward"] = t.ones(ld, dtype=dt, device=dev)      # uint16 counter: never written, 1.0 on every step (:207-212)
        b["done"] = t.zeros(ld, dtype=t.uint8, device=dev)
        b["truncated"] = t.zeros(ld, dtype=t.uint8, device=dev)
        b["action"] = t.zeros(ld, dtype=t.uint8, device=dev)
        b["stats"] = t.tensor([0.0, 0.0, 0.0, math.inf, -math.inf, 0.0], dtype=t.float64, device=dev)
        b["obs"] = t.zeros((4, ld), dtype=dt, device=dev) if self.noisy else None
        tiles = -(-n // _lib.TILE_ENVS[self._dtype_name])
        b["progress"] = t.zeros(2 * tiles, dtype=t.int32, device=dev) if self.tile_ordering else None
        b["env"] = None
        self._buffers = b
        self._refresh_env_struct()
        return b

    def _refresh_env_struct(self):
        b = self._buffers
        env = _lib.CartpoleEnv()
        env.state, env.xi = b["state"].data_ptr(), b["xi"].data_ptr()
        env.elapsed = b["elapsed"].data_ptr() if b["elapsed16"] is None else None
        env.elapsed16 = b["elapsed16"].data_ptr() if b["elapsed16"] is not None else None
        env.beyond = b["beyond"].data_ptr()
        env.progress = b["progress"].data_ptr() if b["progress"] is not None else None
        env.episode = b["episode"].data_ptr() if self.track_episodes else None
        env.n, env.ld = self.num_envs, b["ld"]
        env.env_id0, env.seed = self.env_id0, self._seed
        b["env"] = env
        b["step_plan"] = None          # holds byref(env): rebuild
        b["noise"] = None
        if self.noisy:
            b["noise"] = _lib.ObsNoise()
            b["noise"].obs, b["noise"].std = b["obs"].data_ptr(), math.sqrt(self.noise_level)

    def _resolve(self, name):
        """(C function, leading arguments) of the entry point ``name`` ("reset", "step", "rollout_mlp", ...) for this
        env: the _logged variant while an episode log is attached, the _noisy one for a noisy env, else the plain
        one, each for the env's dtype."""
        b = self._buffers
        head = (ctypes.byref(b["env"]),)
        suffix = "f32" if self._dtype_name == "float32" else "f64"
        if self._episode_log is not None and name in _LOGGED_ENTRIES:
            self._check_log_supported()
            return "renv_cartpole_%s_logged_%s" % (name, suffix), head + (ctypes.byref(self._episode_log.struct),)
        if self.noisy and name in _NOISY_ENTRIES:
            b["noise"].std = math.sqrt(self.noise_level)      # noise_level is a plain attribute in the reference
            return "renv_cartpole_%s_noisy_%s" % (name, suffix), head + (ctypes.byref(b["noise"]),)
        return "renv_cartpole_%s_%s" % (name, suffix), head

    def _scen_what(self):
        return "a scenario mixture" if "table" in self._scen else "per-env scenarios"

    def _resolve_scen(self, name):
        """(C function, leading arguments) of the per-env scenario or mixture form of ``name`` ("reset", "step",
        "rollout", "rollout_mlp", "collect_mlp"): env, scenarios or mixture and -- except for reset -- the episode log
        or NULL."""
        if self.noisy or self._dtype_name != "float32":
            raise ValueError("%s need%s a float32 env without observation noise"
                             % (self._scen_what(), "s" if "table" in self._scen else ""))
        head = (ctypes.byref(self._buffers["env"]), ctypes.byref(self._scen["struct"]))
        if name != "reset":
            if self._episode_log is not None:
                self._check_log_supported()
            head += (ctypes.byref(self._episode_log.struct) if self._episode_log is not None else None,)
        return "renv_cartpole_%s_%s_f32" % (name, "mix" if "table" in self._scen else "scen"), head

    def _launch(self, fn, *args):
        """Call the C function ``fn`` with ``args`` on the env's device and current stream (the last argument)."""
        dev = self._buffers["device"]
        with _device.torch().cuda.device(dev):
            _lib.call(fn, *args, _device.stream_ptr(dev))

    def _integrator(self):
        return _lib.EULER if self.kinematics_integrator == "euler" else _lib.SEMI_IMPLICIT   # :187-196

    def _on_distribution_change(self):
        self._cfg_cache = None

    def _active_dr_cfg(self):
        """DR config used on reset: only when dr_training is on and a distribution is loaded."""
        if not self.dr_training or self.sampling is None:
            return None
        # the reference reads min/max/mean/stdev_task at every draw, so in-place edits of those arrays must take
        # effect: the cached struct is keyed by their bytes (4 x 32 B, ~1 us)
        key = (self.sampling, self.min_task.tobytes(), self.max_task.tobytes(), self.mean_task.tobytes(),
               self.stdev_task.tobytes(),
               np.asarray(self.cov_task).tobytes() if self.sampling == "fullgaussian" else None)
        if self._cfg_cache is None or self._cfg_key != key:
            self._cfg_cache, self._cfg_key = self.dr_config(), key
        return ctypes.byref(self._cfg_cache)

    # ---- gym-style API ------------------------------------------------------------------------------
    def seed(self, seed=None):
        """Philox key for initial states and DR draws (random_cartpole.py:168-170 returns [seed])."""
        if seed is None:
            seed = int(np.random.SeedSequence().entropy % (2 ** 63))
        self._seed = int(seed) & 0xFFFFFFFFFFFFFFFF
        self.seed_dr(self._seed)
        self._tick = 0                  # the reference rebuilds np_random: seed(s); reset() repeats the same episode
        if self._buffers is not None:
            self._refresh_env_struct()
        return [seed]

    def reset(self, mask=None):
        """Reset every env (or those with mask[i] != 0).  Returns obs (N, 4)."""
        b = self._alloc()
        t = _device.torch()
        mask_ptr = None
        if mask is not None:
            mask = t.as_tensor(mask, device=b["device"]).to(t.uint8).contiguous()
            assert mask.shape == (self.num_envs,)
            mask_ptr = _device.ptr(mask)
        viol = self._violation_counter(b["device"])
        if self._scen is not None:
            fn, head = self._resolve_scen("reset")
            self._launch(fn, *head, mask_ptr, self._tick, _device.ptr(viol))
        else:
            fn, head = self._resolve("reset")
            self._launch(fn, *head, mask_ptr, self._tick, self._active_dr_cfg(), _device.ptr(viol))
        self._tick += 1
        return self.obs

    @property
    def obs(self):
        """(N, 4) view of the last observation: the state itself, or the noisy copy for the Noisy variant."""
        b = self._alloc()
        return (b["obs"] if self.noisy else b["state"])[:, :self.num_envs].t()

    @property
    def state(self):
        """(N, 4) view of the true state (what the dynamics integrate; equals ``obs`` unless ``noisy``)."""
        return self._alloc()["state"][:, :self.num_envs].t()

    def _stage_actions(self, actions):
        b = self._buffers
        t = _device.torch()
        n = self.num_envs
        if isinstance(actions, t.Tensor) and actions.is_cuda and actions.dtype == t.uint8 and actions.is_contiguous() \
                and actions.data_ptr() % 16 == 0 and actions.device == b["device"] \
                and (tuple(actions.shape) == (n,) or actions is b["action"]):
            return actions              # zero copy; values outside {0, 1} are flagged by the step kernel itself
        src = actions if isinstance(actions, t.Tensor) else t.as_tensor(np.asarray(actions))
        if tuple(src.shape) != (n,):
            raise ValueError("actions must have shape (%d,), got %s" % (n, tuple(src.shape)))
        if src.dtype.is_floating_point:
            raise AssertionError("%r (%s) invalid" % (actions, type(actions)))   # Discrete(2) rejects floats
        if src.dtype == t.bool:         # a comparison result, e.g. (obs[:, 2] > 0): 0 / 1 by construction
            src = src.to(t.uint8)
        elif src.dtype != t.uint8:
            # a wider integer would be truncated to 8 bits by the staging copy: clamp so that anything outside
            # {0, 1} stays outside (negative -> 255, large -> 255) and is caught on the device
            src = src.to(b["device"], non_blocking=True)
            src = t.where((src < 0) | (src > 255), t.full_like(src, 255), src)
        b["action"][:n].copy_(src, non_blocking=True)
        return b["action"]

    def _step_plan(self):
        """Everything about a ``step`` launch that does not change between calls: the bound C function, the ctypes
        pointers of the persistent buffers and the views handed back.  Rebuilt when a layout-affecting attribute
        changes.  (A 2^20-env step is an 11 us kernel: per-call Python work has to stay below that.)"""
        b = self._buffers
        key = (self.noisy, self.track_truncated, self._dtype_name, self.lean, self._episode_log, self.auto_reset,
               self.max_episode_steps, self._scen_version)
        plan = b.get("step_plan")
        if plan is not None and plan["key"] == key:
            return plan
        self._check_counter()
        t = _device.torch()
        n = self.num_envs
        counter16 = b["elapsed16"] is not None
        # the uint16 counter: the lean step, or with a log attached the logged step on that counter without a reward store
        scen = self._scen is not None
        if scen and not self.auto_reset:
            if "table" in self._scen:
                raise ValueError("a scenario mixture acts at resets: step() with a mixture needs auto_reset")
            raise ValueError("per-env scenarios act at resets: step() with scenarios needs auto_reset")
        if scen:        # one entry point for every layout: the counter of the env, reward NULL with the uint16 one
            fn, head = self._resolve_scen("step")
        else:
            fn, head = self._resolve("step_lean" if counter16 and self._episode_log is None else "step")
        info = {"TimeLimit.truncated": b["truncated"][:n].view(t.bool)} if self.track_truncated else {}
        viol = self._violation_counter(b["device"])
        plan = dict(key=key, fn=getattr(_lib.load(), fn), name=fn, head=head, logged=self._episode_log is not None,
                    lean=counter16 and self._episode_log is None, scen=scen,
                    reward=None if counter16 else _device.ptr(b["reward"]), done=_device.ptr(b["done"]),
                    truncated=_device.ptr(b["truncated"]) if self.track_truncated else None,
                    out=(self.obs, b["reward"][:n], b["done"][:n].view(t.bool)), info=info,
                    device_index=b["device"].index, viol=ctypes.c_void_p(viol.data_ptr()), viol_tensor=viol,
                    own_action=b["action"], own_action_ptr=_device.ptr(b["action"]))
        b["step_plan"] = plan
        return plan

    def step(self, actions):
        """One env-step for all N envs.  actions: (N,) integer tensor/array in {0, 1}.

        Returns (obs (N, 4), reward (N,), done (N,) bool, info) -- views of the env's own buffers, refreshed in place
        by every step (as the reference's obs aliases its state, random_cartpole.py:224).

        Nothing here synchronises with the GPU, so the two errors the reference raises from inside ``step`` /
        ``reset`` -- an action outside Discrete(2) (random_cartpole.py:173-174) and a gaussian DR draw that stayed
        below 0.1 three times (random_env.py:181-186) -- are detected by the kernels, counted on the device and raised
        by the next call that already synchronises: ``step_host_wait``, ``episode_stats``, ``state_dict``,
        ``set_random_task``, ``sample_tasks`` or an explicit ``check_dr_violations()``."""
        b = self._alloc()
        t = _device.torch()
        plan = self._step_plan()
        if actions is plan["own_action"] or actions is b.get("action_view"):   # sample_actions(): nothing to check or copy
            action_ptr = plan["own_action_ptr"]
        else:
            action_ptr = ctypes.c_void_p(self._stage_actions(actions).data_ptr())
        if self.noisy:
            b["noise"].std = math.sqrt(self.noise_level)
        idx = plan["device_index"]
        if plan["scen"]:
            args = plan["head"] + (action_ptr, plan["reward"], plan["done"], plan["truncated"], self._integrator(),
                                   self.max_episode_steps, self._tick, plan["viol"], ctypes.c_void_p(_device.raw_stream(idx)))
        elif plan["lean"]:
            args = plan["head"] + (action_ptr, plan["done"], plan["truncated"], self._integrator(), self.max_episode_steps,
                                   self._tick, self._active_dr_cfg(), plan["viol"], ctypes.c_void_p(_device.raw_stream(idx)))
        elif plan["logged"]:        # auto-reset is implied
            args = plan["head"] + (action_ptr, plan["reward"], plan["done"], plan["truncated"],
                                   self._integrator(), self.max_episode_steps, self._tick,
                                   self._active_dr_cfg(), plan["viol"], ctypes.c_void_p(_device.raw_stream(idx)))
        else:
            args = plan["head"] + (action_ptr, plan["reward"], plan["done"], plan["truncated"],
                                   self._integrator(), self.max_episode_steps, int(self.auto_reset), self._tick,
                                   self._active_dr_cfg(), plan["viol"], ctypes.c_void_p(_device.raw_stream(idx)))
        if t.cuda.current_device() == idx:
            rc = plan["fn"](*args)
        else:
            with t.cuda.device(b["device"]):
                rc = plan["fn"](*args)
        if rc != _lib.OK:
            raise _lib.RenvError(plan["name"], rc, _lib.strerror(rc))
        self._tick += 1
        obs, reward, done = plan["out"]
        return obs, reward, done, dict(plan["info"])

    def _own_action_view(self):
        """(N,) view of the env's own action buffer -- one cached object, recognised by ``step`` without any checks."""
        b = self._buffers
        v = b.get("action_view")
        if v is None:
            v = b["action_view"] = b["action"][:self.num_envs]
        return v

    def sample_actions(self, out=None):
        """``action_space.sample()`` for every env: (N,) uint8 Bernoulli(1/2), Philox keyed by the step clock."""
        b = self._alloc()
        out = b["action"] if out is None else out
        self._launch("renv_random_actions_u8", _device.ptr(out), self.num_envs, self.env_id0, self._seed,
                     self._tick & 0xFFFFFFFF)
        return self._own_action_view() if out is b["action"] else out

    def _check_mlp_supported(self, policy, what):
        if not isinstance(policy, MLPPolicy):
            raise TypeError("%s takes an MLPPolicy (MLPPolicy.from_module(net, device))" % what)
        if self._dtype_name != "float32" or self.noisy:
            raise ValueError("%s with an MLPPolicy needs a float32 env without observation noise" % what)
        if policy.device != self._alloc()["device"]:
            raise ValueError("the MLPPolicy lives on %s, the env on %s" % (policy.device, self._buffers["device"]))

    def policy_actions(self, policy, return_logits=False, *, sample=False, return_logp=False):
        """The actions of ``policy`` (an MLPPolicy) for the current observations of every env, written into the env's
        own action buffer: the returned (N,) uint8 view goes to ``step`` without a copy or a check, as
        ``sample_actions()``'s does.  By default the action is argmax(l0, l1); with ``sample=True`` it is drawn from
        softmax(l0, l1) with the Philox stream of the env's current step clock, i.e. of the ``step`` it goes to
        (include/renv.h renv_cartpole_policy_logp_mlp_f32).  Returns ``actions``, then ``logits`` (N, 2) float32
        (row i = (l0, l1) of env i) with ``return_logits``, then ``logp`` (N,) float32 = log pi(action | obs) with
        ``return_logp``; the tensors are overwritten by the next call.  A fused ``rollout(policy, K)`` equals K x
        step(policy_actions(policy)) bit for bit, and ``collect(policy, K, sample)`` records K x
        step(policy_actions(policy, sample=sample, return_logp=True))."""
        self._check_mlp_supported(policy, "policy_actions()")
        b = self._buffers
        t = _device.torch()
        n = self.num_envs
        logits = logp = None
        if return_logits:
            logits = b.get("mlp_logits")
            if logits is None:
                logits = b["mlp_logits"] = t.empty((2, b["ld"]), dtype=t.float32, device=b["device"])
        if return_logp:
            logp = b.get("mlp_logp")
            if logp is None:
                logp = b["mlp_logp"] = t.empty(b["ld"], dtype=t.float32, device=b["device"])
        if sample or return_logp:
            fn, head = self._resolve("policy_logp_mlp")
            self._launch(fn, *head, ctypes.byref(policy.struct), int(bool(sample)), self._tick, _device.ptr(b["action"]),
                         _device.ptr(logp), _device.ptr(logits))
        else:
            fn, head = self._resolve("policy_actions_mlp")
            self._launch(fn, *head, ctypes.byref(policy.struct), _device.ptr(b["action"]), _device.ptr(logits))
        out = (self._own_action_view(),) + ((logits[:, :n].t(),) if return_logits else ()) + \
            ((logp[:n],) if return_logp else ())
        return out if len(out) > 1 else out[0]

    def trajectory_buffer(self, capacity, logp=True, final_obs=True):
        """A ``Trajectory`` of up to ``capacity`` steps of this env's N envs for ``collect(..., out=buf)``: allocate it
        once and reuse it (2^20 envs x 256 steps with final_obs is ~10 GB).  ``logp`` / ``final_obs`` False: those
        fields are neither allocated nor written."""
        b = self._alloc()
        return Trajectory(self.num_envs, b["ld"], capacity, b["device"], logp=logp, final_obs=final_obs)

    def collect(self, policy, num_steps, sample=True, out=None):
        """``num_steps`` fused env-steps under ``policy`` (an MLPPolicy), recording every step: returns a
        ``Trajectory`` (``out``, or a new buffer when None) with obs, actions, logp, dones, truncated and final_obs
        of each step.  ``sample=True`` draws a ~ softmax(l0, l1) (on-policy data for PPO / A2C-style training),
        ``sample=False`` takes argmax and leaves the env, statistics and episode log exactly as ``rollout(policy, K)``.
        One kernel; bit for bit the K x {obs; policy_actions(policy, sample=sample, return_logp=True); step} loop.
        Advances the step clock by K; afterwards ``obs`` is the observation after the last step (the bootstrap
        observation).  float32 envs without observation noise, and not lean=True."""
        buf = self._alloc()
        if self.lean:
            raise ValueError("collect() keeps the int32 TimeLimit counter: build the env without lean=True")
        self._check_counter()
        self._check_mlp_supported(policy, "collect()")
        K = int(num_steps)
        if K < 1:
            raise ValueError("num_steps must be >= 1, got %d" % K)
        if out is None:
            out = self.trajectory_buffer(K)
        elif not isinstance(out, Trajectory) or out.num_envs != self.num_envs or out.ld != buf["ld"] \
                or out.device != buf["device"]:
            raise ValueError("out is not a trajectory buffer of this env's shape and device: use trajectory_buffer()")
        elif out.capacity < K:
            raise ValueError("out holds %d steps, collect() was asked for %d" % (out.capacity, K))
        viol = self._violation_counter(buf["device"])
        if self._scen is not None:
            fn, head = self._resolve_scen("collect_mlp")
            self._launch(fn, *head, ctypes.byref(policy.struct), ctypes.byref(out.struct), int(bool(sample)), K,
                         self._integrator(), self.max_episode_steps, self._tick, _device.ptr(self._scen["stats"]),
                         _device.ptr(viol))
        else:
            fn, head = self._resolve("collect_mlp")
            self._launch(fn, *head, ctypes.byref(policy.struct), ctypes.byref(out.struct), int(bool(sample)), K,
                         self._integrator(), self.max_episode_steps, self._tick, self._active_dr_cfg(),
                         _device.ptr(buf["stats"]), _device.ptr(viol))
        out.tick0, out.num_steps = self._tick, K
        self._tick += K
        return out

    def gae(self, traj, critic, gamma=0.99, lam=0.95):
        """Values, GAE(gamma, lam) advantages and returns of ``traj``, the trajectory this env's last ``collect`` wrote,
        under ``critic`` (a 1-output MLPPolicy, V(s) = its head): one kernel on the env's stream, which fills
        ``traj.values``, ``traj.advantages`` and ``traj.returns`` ((K, N) float32) and returns ``traj``.

        The reward is 1 on every step.  A terminated step bootstraps nothing, a truncated one bootstraps from
        V(final_obs), and both cut the trace; the last step bootstraps from V(obs), the observation after it.  gamma
        and lam are rounded to float32 and must lie in [0, 1]; the recurrence is that of include/renv.h
        ``renv_cartpole_gae_mlp_f32``.  Raises ValueError unless the env's clock stands where that collect left it
        (any step, reset, rollout or collect since then moved it); a ``set_state()`` in between is not detected and is
        the caller's responsibility.  ``traj`` must have been made with ``final_obs=True``."""
        self._check_mlp_supported(critic, "gae()")
        if critic.outputs != 1:
            raise ValueError("gae() takes a 1-output critic V(s), got a %d-output net" % critic.outputs)
        b = self._buffers
        if not isinstance(traj, Trajectory) or traj.num_envs != self.num_envs or traj.ld != b["ld"] \
                or traj.device != b["device"]:
            raise ValueError("traj is not a trajectory buffer of this env's shape and device")
        if traj._final_obs is None:
            raise ValueError("gae() bootstraps truncated episodes from final_obs: use trajectory_buffer(final_obs=True)")
        if traj.num_steps == 0:
            raise ValueError("traj holds no collected steps")
        g, lm = np.float32(gamma), np.float32(lam)
        if not (0 <= g <= 1 and 0 <= lm <= 1):
            raise ValueError("gamma and lam must lie in [0, 1], got %r and %r" % (gamma, lam))
        if traj.tick0 + traj.num_steps != self._tick:
            raise ValueError("the env has moved since this trajectory was collected (clock %d, the collect ended at %d): "
                             "obs is no longer the observation after its last step" % (self._tick,
                                                                                       traj.tick0 + traj.num_steps))
        values, advantages, returns = traj._gae_storage()
        fn, head = self._resolve("gae_mlp")
        self._launch(fn, *head, ctypes.byref(critic.struct), ctypes.byref(traj.struct), traj.num_steps, float(g), float(lm),
                     _device.ptr(values), _device.ptr(advantages), _device.ptr(returns))
        traj._gae_done()
        return traj

    def rollout(self, w, b=0.0, num_steps=MAX_EPISODE_STEPS):
        """K fused env-steps under the in-kernel linear policy a = [w.s + b > 0] (auto-reset always on), with
        ``w=None`` under the random policy ``action_space.sample()`` (test_random_policy.py:26), or with an
        ``MLPPolicy`` in place of ``w`` under that network (float32 envs without observation noise; ``b`` must be 0)."""
        buf = self._alloc()
        if self.lean:
            raise ValueError("rollout() keeps the int32 TimeLimit counter: build the env without lean=True")
        self._check_counter()
        if isinstance(w, MLPPolicy):
            self._check_mlp_supported(w, "rollout()")
            if float(b) != 0.0:
                raise ValueError("an MLPPolicy carries its own biases: rollout(policy) takes no b")
            name, policy_args = "rollout_mlp", (ctypes.byref(w.struct),)
        else:
            if w is None and self.noisy:        # random policy: the fused equivalent of K x step(sample_actions())
                raise ValueError("the random policy ignores observations: use a noise-free env")
            w_arr = None if w is None else (ctypes.c_double * 4)(*[float(v) for v in w])
            name, policy_args = "rollout", (w_arr, float(b))    # Noisy variant: the policy acts on the noisy observation
        viol = self._violation_counter(buf["device"])
        if self._scen is not None:
            fn, head = self._resolve_scen(name)
            self._launch(fn, *head, *policy_args, int(num_steps), self._integrator(), self.max_episode_steps, self._tick,
                         _device.ptr(self._scen["stats"]), _device.ptr(viol))
        else:
            fn, head = self._resolve(name)
            self._launch(fn, *head, *policy_args, int(num_steps), self._integrator(), self.max_episode_steps, self._tick,
                         self._active_dr_cfg(), _device.ptr(buf["stats"]), _device.ptr(viol))
        self._tick += int(num_steps)

    def evaluate_population(self, policies, num_steps=MAX_EPISODE_STEPS):
        """Evaluate P policies on this env's tasks with common random numbers, in one kernel: ``policies`` is an
        ``MLPPopulation`` or a float32 (P, 5) tensor of linear policies (w0, w1, w2, w3, b: a = [w.s + b > 0]) on the
        env's device.  Returns a (P, 6) float64 device tensor: row p holds the statistics of member p's finished
        episodes (``distributed.STAT_NAMES``, as ``stats_tensor``).

        Member p runs what a fresh twin of this env (same seed, env_id0, task table, DR config, integrator and
        TimeLimit) would run under ``reset()`` then ``rollout(policy_p, num_steps)`` on zeroed statistics, and its row
        equals that twin's ``stats_tensor`` bit for bit: every member sees the same initial states and tasks, so
        differences between rows come from the policies alone.  A row does not depend on P or on the member's
        position.  The env itself is left untouched -- state, tasks, TimeLimit counters, episode counters, statistics,
        an attached episode log -- except for its step clock, which advances by ``num_steps + 1`` so that the next
        call draws new tasks and initial states.  A gaussian DR failure is raised by the next synchronising call, as
        for ``rollout``.  float32 envs without observation noise only."""
        b = self._alloc()
        t = _device.torch()
        if self._scen is not None:
            raise ValueError("evaluate_population() runs the env's own DR config or task table, which %s "
                             "replace%s: call set_scenarios(None) first, or use evaluate_grid()"
                             % (self._scen_what(), "s" if "table" in self._scen else ""))
        K, rows, P, kind, policy_args = self._population_rows(policies, num_steps, "evaluate_population()")
        stats = t.tensor([0.0, 0.0, 0.0, math.inf, -math.inf, 0.0], dtype=t.float64, device=b["device"]).repeat(P, 1)
        viol = self._violation_counter(b["device"])
        self._launch("renv_cartpole_population_%s_f32" % kind, ctypes.byref(b["env"]), *policy_args, P, K,
                     self._integrator(), self.max_episode_steps, self._tick, self._active_dr_cfg(), _device.ptr(stats),
                     _device.ptr(viol))
        self._tick += K + 1             # the fresh start at the current tick, then K steps
        return stats

    def evaluate_grid(self, policies, scenarios, num_steps=MAX_EPISODE_STEPS):
        """Evaluate P policies on C task scenarios in one kernel: ``policies`` as for ``evaluate_population``,
        ``scenarios`` a ``Scenarios`` (fixed tasks and / or DR distributions) on the env's device.  Returns a (P, C, 6)
        float64 device tensor: [p, c] holds the statistics of policy p's finished episodes under scenario c
        (``distributed.STAT_NAMES``).

        Cell [p, c] equals, bit for bit, ``evaluate_population(policies)[p]`` of a twin of this env (same seed,
        env_id0, integrator and TimeLimit, and the same step clock) configured with scenario c: for a distribution,
        ``set_dr_distribution`` with it and ``set_dr_training(True)``; for a fixed task, ``set_task`` with it and no
        DR.  Every cell sees the same initial states and, under one law, the same draws, so differences between cells
        come from the policies and the scenarios alone; a cell depends on neither P, C nor its position.  The env's
        own tasks and DR config are not used, and the env is left untouched except for its step clock, which advances
        by ``num_steps + 1``.  A gaussian DR failure is raised by the next synchronising call.  float32 envs without
        observation noise only."""
        from .scenarios import Scenarios
        b = self._alloc()
        t = _device.torch()
        K, rows, P, kind, policy_args = self._population_rows(policies, num_steps, "evaluate_grid()")
        if not isinstance(scenarios, Scenarios):
            raise TypeError("evaluate_grid() takes its scenarios as a Scenarios (Scenarios.tasks / .distributions)")
        if scenarios.device != b["device"]:
            raise ValueError("the scenarios live on %s, the env on %s" % (scenarios.device, b["device"]))
        C = len(scenarios)
        if P * C * self.num_envs >= 1 << 31:
            raise ValueError("P * C * num_envs = %d: a grid launch takes fewer than 2^31 (policy, scenario, env) triples"
                             % (P * C * self.num_envs))
        stats = t.tensor([0.0, 0.0, 0.0, math.inf, -math.inf, 0.0], dtype=t.float64, device=b["device"]).repeat(P * C, 1)
        viol = self._violation_counter(b["device"])
        self._launch("renv_cartpole_grid_%s_f32" % kind, ctypes.byref(b["env"]), *policy_args, P,
                     _device.ptr(scenarios.rows), C, K, self._integrator(), self.max_episode_steps, self._tick,
                     _device.ptr(stats), _device.ptr(viol))
        self._tick += K + 1             # the fresh start at the current tick, then K steps
        return stats.view(P, C, _lib.NUM_STATS)

    def _population_rows(self, policies, num_steps, what):
        """The checks ``evaluate_population`` and ``evaluate_grid`` share: (K, rows, P, "linear" | "mlp", the policy
        arguments of the C entry point before P)."""
        b = self._buffers
        t = _device.torch()
        if self._dtype_name != "float32" or self.noisy:
            raise ValueError("%s needs a float32 env without observation noise" % what)
        K = int(num_steps)
        if K < 1:
            raise ValueError("num_steps must be >= 1, got %d" % K)
        if isinstance(policies, MLPPopulation):
            rows, width = policies.params, PARAM_FLOATS
        elif isinstance(policies, t.Tensor):
            if policies.dtype != t.float32:
                raise ValueError("linear policies must be a float32 (P, 5) tensor, got %s" % policies.dtype)
            rows, width = policies, 5
        else:
            raise TypeError("%s takes an MLPPopulation or a float32 (P, 5) tensor of linear policies" % what)
        if rows.dim() != 2 or rows.shape[0] < 1 or rows.shape[1] != width or rows.dtype != t.float32:
            raise ValueError("the population must be (P >= 1, %d) float32, got %s %s"
                             % (width, tuple(rows.shape), rows.dtype))
        if rows.device != b["device"]:
            raise ValueError("the population lives on %s, the env on %s" % (rows.device, b["device"]))
        rows = rows.contiguous()
        if width == 5:
            return K, rows, int(rows.shape[0]), "linear", (_device.ptr(rows),)
        return K, rows, int(rows.shape[0]), "mlp", (_device.ptr(rows), policies.activation)

    # ---- episode log ----------------------------------------------------------------------------------
    def start_episode_log(self, capacity=1):
        """Attach a fresh, zeroed episode log with ``capacity`` records per env and return it: from now on every
        episode that ends in ``step()`` or ``rollout()`` (and so in ``step_host_*``) writes one record -- its task,
        terminal state, length, truncated flag and step clock (see ``EpisodeLog``).  ``reset()`` abandons running
        episodes without logging them.  Replaces a log attached before.  Plain auto-reset envs only (fp32, fp64)."""
        self._check_log_supported()
        b = self._alloc()
        self._episode_log = EpisodeLog(self.num_envs, b["ld"], capacity, self.torch_dtype, b["device"], self.env_id0)
        return self._episode_log

    def stop_episode_log(self):
        """Detach the episode log: later steps and rollouts write no records.  The EpisodeLog stays readable."""
        if self._episode_log is None:
            self._check_log_supported()
        self._episode_log = None

    def _check_log_supported(self):
        """The logged entry points imply auto-reset and take no noise block: also checked whenever ``_resolve`` picks
        one, since ``auto_reset`` and ``noisy`` are plain attributes a caller may change with a log attached."""
        if self.lean or self.noisy or not self.auto_reset:
            raise ValueError("the episode log needs an auto-reset env without lean=True or observation noise")

    @property
    def episode_log(self):
        """The attached EpisodeLog, or None."""
        return self._episode_log

    @property
    def stats_tensor(self):
        """Device tensor [episodes, sum R, sum R^2, min R, max R, sum length] (float64).  While per-env scenarios are
        set, a new tensor: the env-wide combination of ``scenario_stats()`` and what was accumulated before."""
        b = self._alloc()
        if self._scen is None:
            return b["stats"]
        return _combine_stats(_device.torch().cat([b["stats"].view(1, -1), self._scen["stats"]]))

    def reset_stats(self):
        t = _device.torch()
        self._alloc()["stats"].copy_(t.tensor(_EMPTY_STATS, dtype=t.float64))
        if self._scen is not None:
            self._scen["stats"].copy_(t.tensor(_EMPTY_STATS, dtype=t.float64).expand_as(self._scen["stats"]))

    # ---- per-env task scenarios -----------------------------------------------------------------------
    def set_scenarios(self, scenarios, assignment=None):
        """Give env i the task scenario ``assignment[i]`` of ``scenarios`` (a ``Scenarios`` on the env's device; C
        rows): from now on every reset of env i -- in ``reset()``, the auto-reset of ``step()``, and inside
        ``rollout()`` and ``collect()`` -- takes its task from that row, and rollouts and collect accumulate the
        finished episodes of each scenario's envs into its row of ``scenario_stats()``.  A distribution row draws as a
        twin env with ``set_dr_distribution`` of it and ``set_dr_training(True)`` would; a fixed-task row gives the
        task, as ``set_task`` of it without DR would.  Env i's results depend on its own row only, so several DR
        distributions -- ADR boundaries, a curriculum, a mixture, an empirical task set -- train in one batch.

        ``assignment`` is N integers in [0, C) (a sequence, a numpy array, or a tensor on the CPU or the env's
        device); it is checked here, with one synchronisation, and copied into the env.  While scenarios are set, the
        DR config, ``dr_training`` and the task table do not decide what a reset draws; ``set_random_task`` and
        ``evaluate_population`` are refused.  Running episodes keep their task until their next reset.
        ``set_scenarios(None)`` restores the env's own configuration.  float32 envs without observation noise."""
        from .scenarios import Scenarios
        t = _device.torch()
        if scenarios is None:
            if assignment is not None:
                raise ValueError("set_scenarios(None) takes no assignment")
            self._clear_scenarios()
            return
        # every argument check that needs no device comes first: nothing is allocated for a refused call
        if self._dtype_name != "float32" or self.noisy:
            raise ValueError("per-env scenarios need a float32 env without observation noise")
        if not isinstance(scenarios, Scenarios):
            raise TypeError("set_scenarios() takes its scenarios as a Scenarios (Scenarios.tasks / .distributions)")
        if scenarios.device.type != "cuda":
            raise ValueError("the scenarios live on %s: move them to the env's device" % scenarios.device)
        C = len(scenarios)
        if C > 65535:
            raise ValueError("at most 65535 scenarios, got %d" % C)
        if assignment is None:
            raise ValueError("set_scenarios() needs an assignment: the scenario of each env")
        a = assignment if isinstance(assignment, t.Tensor) else t.as_tensor(np.asarray(assignment))
        if a.dtype.is_floating_point or a.dtype.is_complex or a.dtype == t.bool:
            raise ValueError("the assignment holds integer scenario indices, got %s" % a.dtype)
        if tuple(a.shape) != (self.num_envs,):
            raise ValueError("the assignment must have shape (%d,), got %s" % (self.num_envs, tuple(a.shape)))
        on_device = a.is_cuda
        if not on_device:
            self._check_assignment_range(a, C)
        b = self._alloc()
        for what, dev in (("scenarios", scenarios.device), ("assignment", a.device if on_device else None)):
            if dev is not None and dev != b["device"]:
                raise ValueError("the %s live on %s, the env on %s" % (what, dev, b["device"]))
        a = a.to(b["device"], t.int64)
        if on_device:
            self._check_assignment_range(a, C)          # the one synchronisation
        self._install_scenarios(scenarios.rows.clone(), a.to(t.int32).to(t.int16),
                                t.tensor(_EMPTY_STATS, dtype=t.float64, device=b["device"]).repeat(C, 1))

    @staticmethod
    def _check_assignment_range(a, C):
        t = _device.torch()
        lo, hi = (int(v) for v in t.stack([a.min(), a.max()]).cpu())
        if lo < 0 or hi >= C:
            raise ValueError("scenario indices must lie in [0, %d), got [%d, %d]" % (C, lo, hi))

    def _install_scenarios(self, rows, of_env, stats):
        """Set the env-owned scenario buffers: rows (C, SCENARIO_FLOATS) float32, of_env (N,) int16 holding the uint16
        indices, stats (C, 6) float64 -- all on the env's device and already checked."""
        t = _device.torch()
        b = self._buffers
        self._clear_scenarios()
        idx = t.zeros(b["ld"], dtype=t.int16, device=b["device"])
        idx[:self.num_envs].copy_(of_env)
        rows = rows.contiguous()
        st = _lib.EnvScenarios()
        st.rows, st.of_env, st.C = rows.data_ptr(), idx.data_ptr(), int(rows.shape[0])
        self._scen = dict(rows=rows, of_env=idx, stats=stats.contiguous(), struct=st)
        self._scen_version += 1

    def _clear_scenarios(self):
        """Drop the scenarios, folding their statistics into the env-wide row."""
        if self._scen is not None:
            self._buffers["stats"].copy_(self.stats_tensor)
            self._scen = None
            self._scen_version += 1

    @property
    def scenarios(self):
        """(rows (C, SCENARIO_FLOATS) float32, assignment (N,) int64) of the env's scenarios, or None."""
        if self._scen is None:
            return None
        return self._scen["rows"], self._scen["of_env"][:self.num_envs].to(_device.torch().int64) & 0xFFFF

    def scenario_stats(self):
        """(C, 6) float64 device tensor: row c holds the statistics (``distributed.STAT_NAMES``) of the episodes that
        the envs of scenario c finished inside ``rollout()`` and ``collect()`` since ``set_scenarios`` or
        ``reset_stats()``.  Each row is exact (integer sums, a min and a max); shards combine row by row as
        ``distributed.combine_stats`` combines ranks, and the rows combined are ``stats_tensor``.  Under a mixture,
        row c holds the episodes whose reset drew row c; the episodes that were running when the mixture was installed
        are in ``stats_tensor`` only."""
        if self._scen is None:
            raise ValueError("no scenarios are set (set_scenarios)")
        return self._scen["stats"][:self._scen["rows"].shape[0]]

    # ---- scenario mixtures ------------------------------------------------------------------------------
    def set_scenario_mixture(self, scenarios, weights):
        """Draw the task scenario of every episode from the C rows of ``scenarios`` (a ``Scenarios`` on the env's
        device) with probabilities proportional to ``weights`` (C finite values >= 0 with a positive sum: a sequence,
        a numpy array or a tensor).  From now on every reset of env i at clock tick t -- in ``reset()``, the
        auto-reset of ``step()``, and inside ``rollout()`` and ``collect()`` -- draws its row on the device from
        Philox (seed, id, t, purpose 6) and an alias table, then resets from that row exactly as ``set_scenarios``
        would with that row assigned to env i.  Successive episodes of an env thus run i.i.d. tasks of the mixture:
        ADR boundary sampling (``Scenarios.adr_boundaries`` with weights ``[1 - p_b] + [p_b / 8] * 8``), weighted
        curricula, an empirical task set.  A weight-0 row is never drawn.

        Rollouts and collect accumulate each finished episode into the ``scenario_stats()`` row its reset drew; the
        episodes running now keep their task and count in ``stats_tensor`` only.  ``scenarios`` holds the rows and
        the row of each env's running episode.  Replaces per-env scenarios or an earlier mixture;
        ``set_scenarios(None)`` clears it.  ``set_mixture_weights`` changes the weights alone.  At most one
        synchronisation.  float32 envs without observation noise; ``set_random_task``, ``evaluate_population`` and
        ``step()`` without auto-reset are refused while a mixture is set."""
        from .scenarios import Scenarios
        t = _device.torch()
        if self._dtype_name != "float32" or self.noisy:
            raise ValueError("a scenario mixture needs a float32 env without observation noise")
        if not isinstance(scenarios, Scenarios):
            raise TypeError("set_scenario_mixture() takes its scenarios as a Scenarios (Scenarios.tasks / .distributions)")
        if scenarios.device.type != "cuda":
            raise ValueError("the scenarios live on %s: move them to the env's device" % scenarios.device)
        C = len(scenarios)
        if C > 65535:
            raise ValueError("at most 65535 scenarios, got %d" % C)
        w, table = _mixture_table(weights, C)
        b = self._alloc()
        if scenarios.device != b["device"]:
            raise ValueError("the scenarios live on %s, the env on %s" % (scenarios.device, b["device"]))
        of_env = t.full((self.num_envs,), C, dtype=t.int32, device=b["device"]).to(t.int16)
        self._install_mixture(scenarios.rows.clone(), w, t.from_numpy(table).to(b["device"]), of_env,
                              t.tensor(_EMPTY_STATS, dtype=t.float64, device=b["device"]).repeat(C + 1, 1))

    def set_mixture_weights(self, weights):
        """New weights for the installed mixture (C values, as ``set_scenario_mixture`` takes them): only the alias
        table is rebuilt.  The rows, the row of every running episode and the statistics are kept, so the next resets
        draw from the new weights while running episodes finish under the row they drew.  The per-iteration call of a
        curriculum or ADR loop; at most one synchronisation."""
        if self._scen is None or "table" not in self._scen:
            raise ValueError("no scenario mixture is set (set_scenario_mixture)")
        w, table = _mixture_table(weights, self._scen["rows"].shape[0])
        self._scen["table"].copy_(_device.torch().from_numpy(table))
        self._scen["weights"] = w

    @property
    def scenario_weights(self):
        """The weights of the installed mixture as given (float64 numpy array of C values), or None."""
        if self._scen is None or "table" not in self._scen:
            return None
        return self._scen["weights"].copy()

    def _install_mixture(self, rows, weights, table, of_env, stats):
        """Set the env-owned mixture buffers: rows (C, SCENARIO_FLOATS) float32, weights (C,) float64 numpy, table (C,)
        int64 alias entries, of_env (N,) int16 holding uint16 rows (C: running since before the mixture), stats
        (C + 1, 6) float64 -- all checked, the tensors on the env's device."""
        t = _device.torch()
        b = self._buffers
        self._clear_scenarios()
        idx = t.zeros(b["ld"], dtype=t.int16, device=b["device"])
        idx[:self.num_envs].copy_(of_env)
        rows, table = rows.contiguous(), table.contiguous()
        st = _lib.EnvMixture()
        st.rows, st.table, st.of_env, st.C = rows.data_ptr(), table.data_ptr(), idx.data_ptr(), int(rows.shape[0])
        self._scen = dict(rows=rows, of_env=idx, stats=stats.contiguous(), struct=st, table=table, weights=weights)
        self._scen_version += 1

    def allgather_stats(self, group=None):
        """The per-iteration collective (distributed.allgather_stats) on this env's statistics; like every call that
        synchronises it also surfaces the device-side error flags."""
        from .distributed import allgather_stats
        combined, gathered = allgather_stats(self.stats_tensor, group)
        host = combined.cpu()                   # synchronises
        self.check_dr_violations()
        return host, gathered

    def episode_stats(self):
        from .distributed import summarize_stats
        stats = self.stats_tensor.cpu().numpy()         # synchronises: the deferred device-side errors surface here
        self.check_dr_violations()
        return summarize_stats(stats)

    def check_dr_violations(self):
        """Raise what the reference would have raised inside step()/reset() (see ``step``); ``validate_actions=False``
        silences the invalid-action assertion (the device flag is then cleared unseen)."""
        if not self.validate_actions and self._dr_violations is not None:
            self._dr_violations[_lib.COUNTER_BAD_ACTION] = 0
        RandomEnv.check_dr_violations(self)

    # ---- tasks --------------------------------------------------------------------------------------
    def get_task(self):
        return self._alloc()["xi"][:self.num_envs]

    def set_task(self, *task):
        """set_task(Tensor(N, 4)) for per-env xi, or set_task(g, m_c, m_p, l) to broadcast one task."""
        b = self._alloc()
        t = _device.torch()
        n = self.num_envs
        if len(task) == 1:
            xi = t.as_tensor(task[0], device=b["device"]).to(self.torch_dtype)
            if xi.shape == (4,):
                xi = xi.reshape(1, 4).expand(n, 4)
            if xi.shape != (n, 4):
                raise ValueError("set_task expects (N, 4) or 4 scalars")
            b["xi"][:n].copy_(xi)
        elif len(task) == 4:
            b["xi"][:n].copy_(t.tensor([float(v) for v in task], dtype=self.torch_dtype,
                                       device=b["device"]).reshape(1, 4).expand(n, 4))
        else:
            raise ValueError("set_task expects (N, 4) or 4 scalars")

    def set_random_task(self):
        """Resample xi of every env now (random_env.py:37-39)."""
        if self._scen is not None:
            raise ValueError("set_random_task() draws from the env's own DR config, which %s replace%s: "
                             "call set_scenarios(None) first" % (self._scen_what(), "s" if "table" in self._scen else ""))
        # sample i of the call is keyed by the GLOBAL env id, so a sharded env draws what the unsharded one would
        self.set_task(self.sample_tasks_tensor(self.num_envs, dtype=self.torch_dtype, device=self._alloc()["device"],
                                               sample_id0=self.env_id0))
        self.check_dr_violations()

    # ---- host-buffer entry point (end-to-end path: H2D actions, D2H results) -------------------------
    def host_buffers(self):
        """Pinned host staging buffers (numpy views): write ``action`` in place to skip one host memcpy."""
        b = self._alloc()
        t = _device.torch()
        n = self.num_envs
        h = b.get("host")
        if h is None:
            h = dict(action=t.empty(b["ld"], dtype=t.uint8).pin_memory(),
                     state=t.empty((4, b["ld"]), dtype=self.torch_dtype).pin_memory(),
                     reward=t.empty(b["ld"], dtype=self.torch_dtype).pin_memory(),
                     done=t.empty(b["ld"], dtype=t.uint8).pin_memory(),
                     truncated=t.empty(b["ld"], dtype=t.uint8).pin_memory(),
                     counters=t.zeros(_lib.NUM_COUNTERS, dtype=t.int64).pin_memory())
            # flag bits: [0] done, [1] truncated, ceil(ld / 32) words each (device twin in b["flag_bits"])
            words = (b["ld"] + 31) // 32
            h["flag_bits"] = t.zeros((2, words), dtype=t.int32).pin_memory()
            b["flag_bits"] = t.zeros((2, words), dtype=t.int32, device=b["device"])
            h["flag_bytes"] = h["flag_bits"].numpy().view(np.uint8)          # (2, 4 * words)
            h["np"] = dict(action=h["action"].numpy()[:n], obs=h["state"].numpy()[:, :n].T,
                           reward=h["reward"].numpy()[:n], done=h["done"].numpy()[:n].view(np.bool_),
                           truncated=h["truncated"].numpy()[:n].view(np.bool_))
            h["reward"].fill_(1)      # with auto-reset the reward is 1.0 on every step (:207-212): never copied
            h["stream"] = t.cuda.Stream(device=b["device"])
            h["event"] = t.cuda.Event()
            b["host"] = h
        return h["np"]

    def step_host_async(self, actions=None):
        """Enqueue one host-buffer step (H2D actions -> step kernel -> D2H obs/reward/done[/truncated]) on this
        env's private stream and return immediately; ``step_host_wait`` returns the numpy results.

        ``actions``: numpy/sequence of {0,1} copied into the pinned staging buffer, or None when the caller has
        already written ``host_buffers()['action']``.  Several envs can have steps in flight at once, which
        overlaps one env's device->host transfer with another's host->device transfer and kernel.
        """
        views = self.host_buffers()
        b = self._buffers
        h = b["host"]
        t = _device.torch()
        if actions is not None:
            acts = np.asarray(actions)
            if acts.dtype != np.uint8:
                if acts.dtype.kind not in "iu":
                    raise AssertionError("%r (%s) invalid" % (actions, type(actions)))   # Discrete(2) rejects floats / bools
                acts = np.clip(acts, -1, 2)     # the cast below wraps mod 256: keep invalid values invalid (255 / 2)
            np.copyto(views["action"], acts, casting="unsafe")
        stream = h["stream"]
        stream.wait_stream(t.cuda.current_stream(b["device"]))
        with t.cuda.stream(stream):
            b["action"].copy_(h["action"], non_blocking=True)
            self.step(b["action"])
            h["state"].copy_(b["obs"] if self.noisy else b["state"], non_blocking=True)
            if not self.auto_reset:        # only the steps-beyond-done rule (:213-222) ever yields 0.0
                h["reward"].copy_(b["reward"], non_blocking=True)
            if self.pack_host_flags:
                sp = _device.stream_ptr(b["device"])
                bits = b["flag_bits"]
                _lib.call("renv_pack_flags_u8", _device.ptr(b["done"]), _device.ptr(bits[0]), self.num_envs, sp)
                if self.track_truncated:
                    _lib.call("renv_pack_flags_u8", _device.ptr(b["truncated"]), _device.ptr(bits[1]), self.num_envs, sp)
                    h["flag_bits"].copy_(bits, non_blocking=True)
                else:
                    h["flag_bits"][0].copy_(bits[0], non_blocking=True)
            else:
                h["done"].copy_(b["done"], non_blocking=True)
                if self.track_truncated:
                    h["truncated"].copy_(b["truncated"], non_blocking=True)
            h["counters"].copy_(self._violation_counter(b["device"]), non_blocking=True)    # 16 bytes: the error flags
            h["event"].record(stream)

    def host_bytes_per_step(self):
        """(host->device, device->host) bytes one ``step_host`` moves over PCIe."""
        esize = 4 if self._dtype_name == "float32" else 8
        ld = self._alloc()["ld"]
        flag = 4 * ((ld + 31) // 32) if self.pack_host_flags else ld
        d2h = 4 * ld * esize + flag + (0 if self.auto_reset else ld * esize) + (flag if self.track_truncated else 0) \
            + 8 * _lib.NUM_COUNTERS
        return ld, d2h

    def step_host_wait(self):
        """Block until the last ``step_host_async`` finished -> (obs (N,4), reward, done, truncated) numpy views."""
        h = self._buffers["host"]
        h["event"].synchronize()
        c = h["counters"]
        if int(c[0]) | int(c[1]):          # the device flagged a gaussian failure or an invalid action (see ``step``)
            self.check_dr_violations()
        v = h["np"]
        if self.pack_host_flags:
            n = self.num_envs
            np.copyto(v["done"].view(np.uint8), np.unpackbits(h["flag_bytes"][0], count=n, bitorder="little"))
            if self.track_truncated:
                np.copyto(v["truncated"].view(np.uint8), np.unpackbits(h["flag_bytes"][1], count=n, bitorder="little"))
        return v["obs"], v["reward"], v["done"], v["truncated"]

    def step_host(self, actions):
        """``step`` with HOST buffers: numpy uint8 actions in, numpy (obs, reward, done, truncated) out."""
        self.step_host_async(actions)
        return self.step_host_wait()

    # ---- checkpoint / resume --------------------------------------------------------------------------
    def _tensor_keys(self):
        """The buffers a state_dict holds; the TimeLimit counter goes under the key of the env's layout."""
        return ("state", "xi", "elapsed16" if self._alloc()["elapsed16"] is not None else "elapsed", "episode", "beyond",
                "stats") + (("obs",) if self.noisy else ())

    def state_dict(self):
        """Everything a resumed run needs to continue bit for bit: env buffers, the Philox key and step clock, the DR
        sampler stream (seed_dr seed, call index), the loaded distribution and the dr_training flag."""
        b = self._alloc()
        out = {k: b[k].clone() for k in self._tensor_keys()}     # the device->host free clone still orders after the kernels
        out.update(seed=self._seed, env_id0=self.env_id0, tick=self._tick, num_envs=self.num_envs,
                   dtype=self._dtype_name, lean=self.lean,
                   dr=dict(seed=self._dr_seed, calls=self._dr_calls, sampling=self.sampling, dr_training=self.dr_training,
                           min_task=self.min_task.copy(), max_task=self.max_task.copy(), mean_task=self.mean_task.copy(),
                           stdev_task=self.stdev_task.copy(),
                           cov_task=np.copy(self.cov_task) if getattr(self, "cov_task", None) is not None else None))
        sc = self._scen
        mixture = sc is not None and "table" in sc
        out["scenarios"] = None if sc is None or mixture else dict(rows=sc["rows"].clone(),
                                                                   of_env=sc["of_env"][:self.num_envs].clone(),
                                                                   stats=sc["stats"].clone())
        if mixture:
            out["mixture"] = dict(rows=sc["rows"].clone(), weights=sc["weights"].copy(), table=sc["table"].clone(),
                                  of_env=sc["of_env"][:self.num_envs].clone(), stats=sc["stats"].clone())
        self.check_dr_violations()          # synchronises; a checkpoint must not hide an error the reference raises
        return out

    def load_state_dict(self, sd):
        """Restore a ``state_dict`` of an env of the same size and dtype, whichever TimeLimit counter layout either env
        has (int32 ``elapsed`` or uint16 ``elapsed16``): the counter is converted."""
        if sd["num_envs"] != self.num_envs or sd["dtype"] != self._dtype_name:
            raise ValueError("state_dict is for %d %s envs" % (sd["num_envs"], sd["dtype"]))
        t = _device.torch()
        b = self._alloc()
        counter = sd["elapsed16"].to(t.int32) & 0xFFFF if "elapsed16" in sd else sd["elapsed"]
        if b["elapsed16"] is not None and "elapsed16" not in sd and int(counter.max()) > 0xFFFF:
            if self.lean:       # counted without a TimeLimit: the uint16 counter cannot hold it
                raise ValueError("the state_dict's TimeLimit counters exceed 65535: load it into an env without lean=True")
            b["elapsed"], b["elapsed16"] = t.zeros_like(b["elapsed16"], dtype=t.int32), None
        for k in self._tensor_keys():
            if k == "elapsed16":
                b[k].copy_(counter.to(b[k].device).to(t.int16))
            else:
                b[k].copy_(counter if k == "elapsed" else sd[k])
        self._seed, self.env_id0, self._tick = sd["seed"], sd["env_id0"], sd["tick"]
        dr = sd.get("dr")
        if dr is not None:
            self._dr_seed, self._dr_calls = dr["seed"], dr["calls"]
            self.sampling, self.dr_training = dr["sampling"], dr["dr_training"]
            self.min_task[:], self.max_task[:] = dr["min_task"], dr["max_task"]
            self.mean_task[:], self.stdev_task[:] = dr["mean_task"], dr["stdev_task"]
            if dr["cov_task"] is not None:
                self.cov_task = np.copy(dr["cov_task"])
            self._on_distribution_change()
        self._refresh_env_struct()
        self._scen = None
        self._scen_version += 1
        sc = sd.get("scenarios")
        if sc is not None:
            dev = b["device"]
            self._install_scenarios(sc["rows"].to(dev), sc["of_env"].to(dev), sc["stats"].to(dev).clone())
        mx = sd.get("mixture")
        if mx is not None:
            dev = b["device"]
            # clones: set_mixture_weights rewrites the table in place, which must not reach the caller's state_dict
            self._install_mixture(mx["rows"].to(dev).clone(), np.array(mx["weights"], dtype=np.float64),
                                  mx["table"].to(dev).clone(), mx["of_env"].to(dev), mx["stats"].to(dev).clone())

    # ---- introspection used by tests -------------------------------------------------------------------
    @property
    def elapsed(self):
        b = self._alloc()
        if b["elapsed16"] is not None:
            t = _device.torch()
            return b["elapsed16"][:self.num_envs].to(t.int32) & 0xFFFF
        return b["elapsed"][:self.num_envs]

    @property
    def episode(self):
        return self._alloc()["episode"][:self.num_envs]

    @property
    def steps_beyond_done(self):
        return self._alloc()["beyond"][:self.num_envs]

    def set_state(self, state, elapsed=None):
        """Inject per-env states (N, 4) (parity tests: the reference's ``env.state = s0``)."""
        b = self._alloc()
        t = _device.torch()
        st = t.as_tensor(state, device=b["device"]).to(self.torch_dtype)
        b["state"][:, :self.num_envs].copy_(st.t())
        b["beyond"].fill_(-1)
        if elapsed is not None:
            el = t.as_tensor(elapsed, device=b["device"]).to(t.int32)
            if b["elapsed16"] is not None:
                b["elapsed16"][:self.num_envs].copy_(el.to(t.int16))
            else:
                b["elapsed"][:self.num_envs].copy_(el)
