"""Per-step trajectory buffer of ``RandomCartPoleVecEnv.collect`` (include/renv.h ``renv_trajectory``).

    buf = venv.trajectory_buffer(256)                    # allocate once, reuse every training iteration
    traj = venv.collect(policy, 256, out=buf)           # one kernel: K steps under a ~ softmax(policy logits)
    traj.obs, traj.actions, traj.logp, traj.dones, traj.truncated, traj.final_obs, traj.rewards

Step k of env i is row ``[k, i]`` of every field: ``obs`` is the observation the action was chosen from, ``logp`` is
``log pi(action | obs)``, ``dones`` / ``truncated`` are what ``step()`` returned for that step, and ``final_obs`` holds,
where ``dones``, the observation after the step that auto-reset replaced (the value to bootstrap a truncated episode
from; elsewhere it is stale).  After ``collect`` the env's ``obs`` is the observation that follows the last step.

    venv.gae(traj, critic, gamma=0.99, lam=0.95)         # one kernel: V under a 1-output MLPPolicy, GAE, returns
    traj.values, traj.advantages, traj.returns

``gae`` fills ``values`` (V(obs[k])), ``advantages`` and ``returns`` (``advantages + values``), each (K, N) float32;
they are None until ``gae()`` has run on the current collect.
"""
from . import _device, _lib


class Trajectory:
    """Device buffers of up to ``capacity`` steps of ``num_envs`` envs, and the views of the steps last collected."""

    def __init__(self, num_envs, ld, capacity, device, logp=True, final_obs=True):
        t = _device.torch()
        capacity = int(capacity)
        if not 1 <= capacity <= 0x7FFFFFFF:
            raise ValueError("trajectory capacity must be in [1, 2^31 - 1], got %d" % capacity)
        self.num_envs, self.ld, self.capacity, self.device = int(num_envs), int(ld), capacity, t.device(device)
        self._obs = t.empty((capacity, ld, 4), dtype=t.float32, device=device)
        self._action = t.empty((capacity, ld), dtype=t.uint8, device=device)
        self._done = t.empty((capacity, ld), dtype=t.uint8, device=device)
        self._truncated = t.empty((capacity, ld), dtype=t.uint8, device=device)
        self._logp = t.empty((capacity, ld), dtype=t.float32, device=device) if logp else None
        self._final_obs = t.zeros((capacity, ld, 4), dtype=t.float32, device=device) if final_obs else None
        s = _lib.Trajectory()
        s.obs, s.action, s.done, s.truncated = (self._obs.data_ptr(), self._action.data_ptr(), self._done.data_ptr(),
                                                self._truncated.data_ptr())
        s.logp = self._logp.data_ptr() if logp else None
        s.final_obs = self._final_obs.data_ptr() if final_obs else None
        s.capacity = capacity
        self.struct = s
        self._values = self._advantages = self._returns = None      # (capacity, ld) float32, allocated by gae()
        self.tick0 = None           # step clock of step 0 of the last collect
        self.num_steps = 0          # steps the last collect wrote

    @property
    def tick0(self):
        """Step clock of step 0 of the last collect (None before the first)."""
        return self._tick0

    @tick0.setter
    def tick0(self, tick):
        self._tick0 = tick
        self._gae_tick0 = None      # a new collect (even one at the same clock, after seed()): the values, advantages
                                    # and returns no longer belong to the data

    def _gae_storage(self):
        """The (capacity, ld) value / advantage / return arrays, allocated on the first ``gae()`` and then reused."""
        if self._values is None:
            t = _device.torch()
            self._values, self._advantages, self._returns = (
                t.empty((self.capacity, self.ld), dtype=t.float32, device=self.device) for _ in range(3))
        return self._values, self._advantages, self._returns

    def _gae_done(self):
        """Record that ``gae()`` has filled the arrays for the current collect."""
        self._gae_tick0 = self._tick0

    def _view(self, buf):
        return None if buf is None else buf[:self.num_steps, :self.num_envs]

    def _gae_view(self, buf):
        return self._view(buf) if self._gae_tick0 is not None else None

    @property
    def values(self):
        """(K, N) float32 V(obs[k]) of the critic of the last ``gae()``, or None unless ``gae()`` ran on this collect."""
        return self._gae_view(self._values)

    @property
    def advantages(self):
        """(K, N) float32 GAE advantages of the last ``gae()``, or None unless ``gae()`` ran on this collect."""
        return self._gae_view(self._advantages)

    @property
    def returns(self):
        """(K, N) float32 ``advantages + values`` (the critic's regression target), or None unless ``gae()`` ran on
        this collect."""
        return self._gae_view(self._returns)

    @property
    def obs(self):
        """(K, N, 4) float32: x, x_dot, theta, theta_dot the action of step k was chosen from."""
        return self._view(self._obs)

    @property
    def actions(self):
        """(K, N) uint8: the action taken at step k."""
        return self._view(self._action)

    @property
    def logp(self):
        """(K, N) float32 log pi(action | obs), or None for a buffer made with ``logp=False``."""
        return self._view(self._logp)

    @property
    def dones(self):
        """(K, N) bool: step k ended the episode (terminated or truncated); the next row starts a new one."""
        return self._view(self._done).view(_device.torch().bool)

    @property
    def truncated(self):
        """(K, N) bool: the TimeLimit ended the episode at step k (``info['TimeLimit.truncated']``)."""
        return self._view(self._truncated).view(_device.torch().bool)

    @property
    def final_obs(self):
        """(K, N, 4) float32: the observation after step k, valid where ``dones`` (the terminal observation auto-reset
        replaced); None for a buffer made with ``final_obs=False``."""
        return self._view(self._final_obs)

    @property
    def rewards(self):
        """(K, N) float32 ones: with auto-reset the reward is 1.0 on every step (random_cartpole.py:207-212).  An
        expanded view: no buffer is stored or written."""
        t = _device.torch()
        return t.ones((), dtype=t.float32, device=self.device).expand(self.num_steps, self.num_envs)
