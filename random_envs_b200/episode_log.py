"""Episode log of a RandomCartPoleVecEnv: one record per episode that ends in ``step()`` or ``rollout()``.

    log = venv.start_episode_log(capacity=4)
    venv.rollout(w, 0.0, 500)
    ep = log.episodes()          # flat tensors: env_id, xi, final_state, length, truncated, end_tick

Each env keeps a ring of ``capacity`` records (include/renv.h ``renv_episode_log``): the record of the ``c``-th episode
env ``i`` ended (``c`` counted from 0) is in slot ``c % capacity``, and ``count[i]`` is the number of episodes it ended
since the log was started or cleared.  A record holds the task the episode ran under (before the resample of its
reset), the state after its last step (the terminal observation auto-reset overwrites), its length (= its return:
the reward is 1.0 on every step), whether the TimeLimit truncated it, and the step clock of its last step.  The
kernels write the records; nothing here runs per step.
"""
from . import _device, _lib


class EpisodeLog:
    """Device buffers of an episode log plus the views and helpers to read them (see the module docstring)."""

    def __init__(self, num_envs, ld, capacity, dtype, device, env_id0=0):
        t = _device.torch()
        capacity = int(capacity)
        if not 1 <= capacity <= 0x7FFFFFFF:
            raise ValueError("episode log capacity must be in [1, 2^31 - 1], got %d" % capacity)
        self.num_envs, self.capacity, self.env_id0 = int(num_envs), capacity, int(env_id0)
        self._xi = t.zeros((capacity, ld, 4), dtype=dtype, device=device)
        self._final_state = t.zeros((capacity, ld, 4), dtype=dtype, device=device)
        self._length = t.zeros((capacity, ld), dtype=t.int32, device=device)
        self._truncated = t.zeros((capacity, ld), dtype=t.uint8, device=device)
        self._end_tick = t.zeros((capacity, ld), dtype=t.int64, device=device)
        self._count = t.zeros(ld, dtype=t.int32, device=device)
        s = _lib.EpisodeLog()
        s.xi, s.final_state = self._xi.data_ptr(), self._final_state.data_ptr()
        s.length, s.truncated = self._length.data_ptr(), self._truncated.data_ptr()
        s.end_tick, s.count = self._end_tick.data_ptr(), self._count.data_ptr()
        s.capacity = capacity
        self.struct = s

    # ---- ring views (slot j of env i = the latest episode c of env i with c % capacity == j) -----------------------
    @property
    def xi(self):
        """(capacity, N, 4): gravity, cart_mass, pole_mass, pole_length the episode ran under."""
        return self._xi[:, :self.num_envs]

    @property
    def final_state(self):
        """(capacity, N, 4): x, x_dot, theta, theta_dot after the step that ended the episode."""
        return self._final_state[:, :self.num_envs]

    @property
    def length(self):
        """(capacity, N) int32: env-steps of the episode, counted across calls (= its return)."""
        return self._length[:, :self.num_envs]

    @property
    def truncated(self):
        """(capacity, N) bool: the TimeLimit ended the episode without meeting the thresholds."""
        return self._truncated[:, :self.num_envs].view(_device.torch().bool)

    @property
    def end_tick(self):
        """(capacity, N) int64: step clock of the step that ended the episode."""
        return self._end_tick[:, :self.num_envs]

    @property
    def count(self):
        """(N,) int32: episodes ended per env since the log was started or cleared."""
        return self._count[:self.num_envs]

    def clear(self):
        """Forget every record (enqueued on the current stream, like the kernels that write them)."""
        for buf in (self._xi, self._final_state, self._length, self._truncated, self._end_tick, self._count):
            buf.zero_()

    def episodes(self):
        """Every logged episode as flat device tensors in (env, chronological) order: ``env_id`` (global, int64),
        ``xi`` (E, 4), ``final_state`` (E, 4), ``length`` (E,) int32, ``truncated`` (E,) bool and ``end_tick`` (E,)
        int64.  Synchronises.  Raises OverflowError when a ring has overwritten records: read the ring views instead,
        or start the log with a larger capacity."""
        t = _device.torch()
        count = self.count.to(t.int64)
        lost = int((count - self.capacity).clamp_(min=0).sum())
        if lost:
            raise OverflowError("episode log overwrote %d episodes (capacity %d per env): start it with a larger "
                                "capacity or read it more often" % (lost, self.capacity))
        # without overwrites slot j of env i holds episode j of env i
        keep = t.arange(self.capacity, device=count.device)[None, :] < count[:, None]          # (N, capacity)
        env_id = (t.arange(self.num_envs, device=count.device, dtype=t.int64) + self.env_id0)[:, None].expand_as(keep)
        per_env = lambda v: v.transpose(0, 1)[keep]                                          # (capacity, N, ...) -> (E, ...)
        return dict(env_id=env_id[keep], xi=per_env(self.xi), final_state=per_env(self.final_state),
                    length=per_env(self.length), truncated=per_env(self.truncated), end_tick=per_env(self.end_tick))
