"""Load the UNMODIFIED reference hot-path source by file path.

TEST INFRASTRUCTURE (see oracle/__init__.py).  The source comes from
``/root/reference`` where that is mounted (the build container) and otherwise
from ``oracle/_ref/`` -- byte-identical copies of the two files made there by
``oracle/make_ref.py`` (git-ignored, shipped to the GPU box with the snapshot)
so that ``bench.py``'s CPU legs can time the real reference on the box's host.
Tests that compare against the live reference skip when neither is present and
rely on the golden vectors this loader produced (``oracle/make_golden.py``).

Why by path: ``import random_envs`` runs ``random_envs/__init__.py:1`` which
imports the MuJoCo sub-package (``jinja/jinja_mujoco_env.py:15-18`` raises
without mujoco_py) before it ever reaches CartPole.  The two hot-path files
``random_envs/random_env.py`` and ``random_envs/random_cartpole.py`` have no
other dependency than gym/numpy/math, so they are exec'd directly under the
gym shim.  Two names the reference forgot to import are injected into the
module namespace (``random_env.py:161,163`` uses ``truncnorm``; ``:236`` uses
``csv``); the source text itself is not touched.
"""
import csv
import importlib.util
import os
import sys
import types

import numpy as np

from . import gym_shim

_HERE = os.path.dirname(os.path.abspath(__file__))


def _has_sources(root):
    return all(os.path.isfile(os.path.join(root, "random_envs", f)) for f in ("random_env.py", "random_cartpole.py"))


def _resolve_root():
    for cand in (os.environ.get("RENV_REFERENCE_ROOT"), "/root/reference", os.path.join(_HERE, "_ref")):
        if cand and _has_sources(cand):
            return cand
    return os.environ.get("RENV_REFERENCE_ROOT", "/root/reference")


REFERENCE_ROOT = _resolve_root()

# skip reason of the tests that compare with the original live: no stored run of the original covers what they compare
UNAVAILABLE = ("needs the original random-envs source, which is not part of this repository; set RENV_REFERENCE_ROOT to "
               "a checkout of gabrieletiboni/random-envs to run this comparison")


def available():
    return _has_sources(REFERENCE_ROOT)


_cache = {}


def load():
    """Return (random_env_module, random_cartpole_module) of the real reference."""
    if "mods" in _cache:
        return _cache["mods"]
    if not available():
        raise FileNotFoundError("reference tree not mounted at %s" % REFERENCE_ROOT)
    saved = {k: sys.modules.get(k) for k in list(sys.modules)
             if k == "gym" or k.startswith("gym.") or k == "random_envs" or k.startswith("random_envs.")}
    gym_shim.install()
    try:
        pkg = types.ModuleType("random_envs")
        pkg.__path__ = []  # a namespace stub: never runs the reference's __init__ (MuJoCo import)
        sys.modules["random_envs"] = pkg
        mods = []
        for name in ("random_env", "random_cartpole"):
            path = os.path.join(REFERENCE_ROOT, "random_envs", name + ".py")
            spec = importlib.util.spec_from_file_location("random_envs." + name, path)
            mod = importlib.util.module_from_spec(spec)
            sys.modules["random_envs." + name] = mod
            spec.loader.exec_module(mod)
            setattr(pkg, name, mod)
            mods.append(mod)
        import scipy.stats
        mods[0].truncnorm = scipy.stats.truncnorm  # missing import, random_env.py:161
        mods[0].csv = csv                          # missing import, random_env.py:236
    finally:
        # leave no fake `gym` / `random_envs` behind for the rest of the process
        for k in [k for k in sys.modules if k == "gym" or k.startswith("gym.")
                  or k == "random_envs" or k.startswith("random_envs.")]:
            del sys.modules[k]
        for k, v in saved.items():
            if v is not None:
                sys.modules[k] = v
    _cache["mods"] = tuple(mods)
    return _cache["mods"]


def make_cartpole():
    """A bare reference ``RandomCartPoleEnv`` (no TimeLimit wrapper)."""
    _, rc = load()
    return rc.RandomCartPoleEnv()


def make_sampler_env(dim, lower_bounds, search_bounds=None):
    """A ``RandomEnv`` subclass with a ``dim``-dimensional xi table.

    MuJoCo envs cannot be instantiated here; the sampler code
    (``random_env.py:148-203``) only needs ``min/max/mean/stdev_task`` and
    ``get_task_lower_bound(i)``, so this carries e.g. the humanoid's 30-dim
    table (``jinja/random_humanoid.py:113-146``) through the reference's own
    ``sample_task``.
    """
    re_mod, _ = load()
    lb = np.asarray(lower_bounds, dtype=np.float64)

    class _TableEnv(re_mod.RandomEnv):
        def __init__(self):
            re_mod.RandomEnv.__init__(self)
            self.task_dim = dim
            self.min_task = np.zeros(dim)
            self.max_task = np.zeros(dim)
            self.mean_task = np.zeros(dim)
            self.stdev_task = np.zeros(dim)
            self._task = np.zeros(dim)

        def get_task_lower_bound(self, index):
            return lb[index]

        def get_search_bounds_mean(self, index):
            return search_bounds[index]

        def get_task(self):
            return self._task.copy()

        def set_task(self, *task):
            self._task = np.array(task, dtype=np.float64)

    return _TableEnv()
