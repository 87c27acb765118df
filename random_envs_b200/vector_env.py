"""Vectorised, tensor-in/tensor-out RandomCartPole: N envs resident in HBM, one kernel per call.

Same method names as the reference's single env (random_cartpole.py / random_env.py): ``reset``,
``step``, ``seed``, ``get_task``, ``set_task``, ``set_random_task``, ``set_dr_distribution``,
``set_dr_training`` ...; arguments and results are batched torch CUDA tensors:

    reset()        -> obs (N, 4)
    step(actions)  -> obs (N, 4), reward (N,), done (N,) bool, info {'TimeLimit.truncated': (N,) bool}
    get_task()     -> (N, 4)            set_task(Tensor(N, 4) | g, m_c, m_p, l)
    rollout(w, b, K) -> None            (K fused steps of the linear policy a = [w.s + b > 0] or of an MLPPolicy)
    evaluate_population(policies, K) -> (P, 6)   (P policies on common tasks from fresh starts; the env is untouched)
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


def _round_up(x, m):
    return (x + m - 1) // m * m


class RandomCartPoleVecEnv(RandomEnv):
    """N domain-randomised cart-poles stepped by hand-written sm_100a kernels."""

    def __init__(self, num_envs, dtype="float32", device=None, seed=0, env_id0=0,
                 max_episode_steps=MAX_EPISODE_STEPS, auto_reset=True, kinematics_integrator="euler",
                 track_truncated=True, validate_actions=True, track_episodes=True, noisy=False, noise_level=1e-4,
                 lean=False, tile_ordering="auto", pack_host_flags=True):
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
        # of 62 bytes of HBM traffic per env-step; state / done / truncated bit-identical
        self.lean = bool(lean)
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
        b["elapsed"] = None if self.lean else t.zeros(ld, dtype=t.int32, device=dev)
        b["elapsed16"] = t.zeros(ld, dtype=t.int16, device=dev) if self.lean else None     # uint16 bit pattern
        b["episode"] = t.zeros(ld, dtype=t.int32, device=dev)       # uint32 bit pattern
        b["beyond"] = t.full((ld,), -1, dtype=t.int32, device=dev)
        b["reward"] = t.ones(ld, dtype=dt, device=dev)      # lean: never written, 1.0 on every step (:207-212)
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
        env.elapsed = None if self.lean else b["elapsed"].data_ptr()
        env.elapsed16 = b["elapsed16"].data_ptr() if self.lean else None
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
        key = (self.noisy, self.track_truncated, self._dtype_name, self.lean, self._episode_log, self.auto_reset)
        plan = b.get("step_plan")
        if plan is not None and plan["key"] == key:
            return plan
        t = _device.torch()
        n = self.num_envs
        fn, head = self._resolve("step_lean" if self.lean else "step")
        info = {"TimeLimit.truncated": b["truncated"][:n].view(t.bool)} if self.track_truncated else {}
        viol = self._violation_counter(b["device"])
        plan = dict(key=key, fn=getattr(_lib.load(), fn), name=fn, head=head, logged=self._episode_log is not None,
                    reward=_device.ptr(b["reward"]), done=_device.ptr(b["done"]),
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
        if self.lean:
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
        observation).  float32 envs without observation noise or lean=True only."""
        buf = self._alloc()
        if self.lean:
            raise ValueError("collect() keeps the int32 TimeLimit counter: build the env without lean=True")
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
        fn, head = self._resolve("collect_mlp")
        viol = self._violation_counter(buf["device"])
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
        fn, head = self._resolve(name)
        viol = self._violation_counter(buf["device"])
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
        if self._dtype_name != "float32" or self.noisy:
            raise ValueError("evaluate_population() needs a float32 env without observation noise")
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
            raise TypeError("evaluate_population() takes an MLPPopulation or a float32 (P, 5) tensor of linear policies")
        if rows.dim() != 2 or rows.shape[0] < 1 or rows.shape[1] != width or rows.dtype != t.float32:
            raise ValueError("the population must be (P >= 1, %d) float32, got %s %s"
                             % (width, tuple(rows.shape), rows.dtype))
        if rows.device != b["device"]:
            raise ValueError("the population lives on %s, the env on %s" % (rows.device, b["device"]))
        rows = rows.contiguous()
        P = int(rows.shape[0])
        stats = t.tensor([0.0, 0.0, 0.0, math.inf, -math.inf, 0.0], dtype=t.float64, device=b["device"]).repeat(P, 1)
        if width == 5:
            fn, policy_args = "renv_cartpole_population_linear_f32", (_device.ptr(rows), P)
        else:
            fn, policy_args = "renv_cartpole_population_mlp_f32", (_device.ptr(rows), policies.activation, P)
        viol = self._violation_counter(b["device"])
        self._launch(fn, ctypes.byref(b["env"]), *policy_args, K, self._integrator(), self.max_episode_steps, self._tick,
                     self._active_dr_cfg(), _device.ptr(stats), _device.ptr(viol))
        self._tick += K + 1             # the fresh start at the current tick, then K steps
        return stats

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
        """Device tensor [episodes, sum R, sum R^2, min R, max R, sum length] (float64)."""
        return self._alloc()["stats"]

    def reset_stats(self):
        t = _device.torch()
        self._alloc()["stats"].copy_(t.tensor([0.0, 0.0, 0.0, math.inf, -math.inf, 0.0], dtype=t.float64))

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
        return ("state", "xi", "elapsed16" if self.lean else "elapsed", "episode", "beyond", "stats") + \
               (("obs",) if self.noisy else ())

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
        self.check_dr_violations()          # synchronises; a checkpoint must not hide an error the reference raises
        return out

    def load_state_dict(self, sd):
        if sd["num_envs"] != self.num_envs or sd["dtype"] != self._dtype_name or sd.get("lean", False) != self.lean:
            raise ValueError("state_dict is for %d %s envs%s" % (sd["num_envs"], sd["dtype"], " (lean)" if sd.get("lean") else ""))
        b = self._alloc()
        for k in self._tensor_keys():
            b[k].copy_(sd[k])
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

    # ---- introspection used by tests -------------------------------------------------------------------
    @property
    def elapsed(self):
        b = self._alloc()
        if self.lean:
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
            if self.lean:
                b["elapsed16"][:self.num_envs].copy_(el.to(t.int16))
            else:
                b["elapsed"][:self.num_envs].copy_(el)
