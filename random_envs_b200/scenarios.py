"""Task scenarios: the columns of an evaluation grid (``RandomCartPoleVecEnv.evaluate_grid``), and the per-env task
configurations of training (``RandomCartPoleVecEnv.set_scenarios``).

A scenario is either a fixed task (gravity, cart_mass, pole_mass, pole_length), kept by every episode, or a DR
distribution that every episode draws its task from.  Each is one row of ``RENV_SCENARIO_FLOATS`` float32 values in
device memory, written by ``renv_scenario_pack_f32`` (include/renv.h): the parameters a launch of the env with that
configuration passes to its kernels, so a grid cell sees exactly the tasks a twin env configured that way would.
"""
import ctypes

import numpy as np

from . import _device, _lib
from .random_env import TaskSampler


def _pack(cfg, task, out):
    """Row ``out`` (a float32 numpy view of SCENARIO_FLOATS values) of the renv_dr_cfg ``cfg`` or of ``task``."""
    task_arg = (ctypes.c_double * 4)(*task) if task is not None else None
    _lib.call("renv_scenario_pack_f32", ctypes.byref(cfg) if cfg is not None else None, task_arg,
              ctypes.c_void_p(out.ctypes.data))


class Scenarios:
    """C scenario rows for ``RandomCartPoleVecEnv.evaluate_grid`` and ``set_scenarios``: ``rows`` is a (C, SCENARIO_FLOATS) float32 tensor on
    ``device``.  Build them with ``Scenarios.tasks`` (fixed tasks) or ``Scenarios.distributions`` (DR distributions)
    and join them with ``Scenarios.cat``.

    The ADR boundary check -- a policy's return with one dim pinned at a boundary of the current ranges and the others
    drawn from them -- is a uniform distribution whose range on that dim has lo = hi: with width 0 the draw is
    fma(0, u, lo) = lo exactly, so the dim is the boundary value in every episode."""

    def __init__(self, rows):
        t = _device.torch()
        if not isinstance(rows, t.Tensor) or rows.dtype != t.float32 or rows.dim() != 2 \
                or rows.shape[1] != _lib.SCENARIO_FLOATS:
            raise ValueError("scenario rows are a (C, %d) float32 tensor" % _lib.SCENARIO_FLOATS)
        if rows.shape[0] < 1:
            raise ValueError("a grid needs at least one scenario")
        self.rows = rows.contiguous()           # 128-byte rows: each 16-byte aligned when the base is
        self.device = self.rows.device

    @staticmethod
    def _place(host, device):
        t = _device.torch()
        dev = _device.require_cuda() if device is None else t.device(device)
        return Scenarios(t.from_numpy(host).to(dev))

    @classmethod
    def tasks(cls, tasks, device=None):
        """Fixed-task rows from a (C, 4) array or tensor of (gravity, cart_mass, pole_mass, pole_length).  Cell (p, c)
        then equals ``evaluate_population`` of a twin env whose every task is row c, without DR."""
        t = _device.torch()
        arr = tasks.detach().to("cpu", t.float64).numpy() if isinstance(tasks, t.Tensor) \
            else np.asarray(tasks, dtype=np.float64)
        if arr.ndim != 2 or arr.shape[0] < 1 or arr.shape[1] != 4:
            raise ValueError("tasks must be a (C >= 1, 4) array, got shape %s" % (arr.shape,))
        if not np.isfinite(arr).all():
            raise ValueError("tasks must be finite")
        host = np.zeros((arr.shape[0], _lib.SCENARIO_FLOATS), dtype=np.float32)
        for c in range(arr.shape[0]):
            _pack(None, arr[c].tolist(), host[c])
        return cls._place(host, device)

    @classmethod
    def distributions(cls, dr_type, distrs, device=None):
        """One DR row per entry of ``distrs``, each given as ``set_dr_distribution(dr_type, distr)`` takes it
        (interleaved pairs, or ``{"mean", "cov"}`` for fullgaussian).  Each row is built by a fresh
        ``TaskSampler("RandomCartPole-v0")``, so the validation and its errors are the env's own, and the row holds
        what a twin env with that distribution and ``set_dr_training(True)`` would launch with."""
        distrs = list(distrs)
        if not distrs:
            raise ValueError("a grid needs at least one scenario")
        host = np.zeros((len(distrs), _lib.SCENARIO_FLOATS), dtype=np.float32)
        for c, distr in enumerate(distrs):
            sampler = TaskSampler("RandomCartPole-v0")
            sampler.set_dr_distribution(dr_type, distr)
            _pack(sampler.dr_config(), None, host[c])
        return cls._place(host, device)

    @classmethod
    def adr_boundaries(cls, low, high, device=None):
        """The 1 + 2 x 4 uniform rows of an ADR iteration over the box [low, high] (two length-4 sequences): row 0 is
        the box itself, row 1 + 2k the box with dim k pinned at ``low[k]`` and row 2 + 2k the box with dim k pinned at
        ``high[k]`` (width 0: see the class docstring).  Built through ``Scenarios.distributions``, so the ranges are
        validated as ``set_dr_distribution("uniform", ...)`` validates them.  How the ranges grow or shrink from the
        returns of each row is left to the caller."""
        lo, hi = np.asarray(low, dtype=np.float64), np.asarray(high, dtype=np.float64)
        if lo.shape != (4,) or hi.shape != (4,):
            raise ValueError("low and high are 4 values each (gravity, cart_mass, pole_mass, pole_length)")
        boxes = [(lo, hi)]
        for k in range(4):
            for v in (lo[k], hi[k]):
                pl, ph = lo.copy(), hi.copy()
                pl[k] = ph[k] = v
                boxes.append((pl, ph))
        return cls.distributions("uniform", [np.stack([pl, ph], 1).reshape(-1).tolist() for pl, ph in boxes], device)

    @classmethod
    def cat(cls, *parts):
        """The scenarios of ``parts`` (Scenarios on one device), in order."""
        if not parts or not all(isinstance(p, Scenarios) for p in parts):
            raise TypeError("Scenarios.cat takes one or more Scenarios")
        if len({p.device for p in parts}) != 1:
            raise ValueError("the scenarios to join live on different devices")
        return cls(_device.torch().cat([p.rows for p in parts]))

    def __len__(self):
        return int(self.rows.shape[0])
