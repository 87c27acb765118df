"""ctypes binding of librenv_b200.so -- the only way the package reaches the GPU.

There is NO fallback: if the library is missing, fails to load, or lacks a symbol declared in
include/renv.h this module raises, and every compute entry point of the package raises with it.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "librenv_b200.so")

ABI_VERSION = 6
MAX_DIM = 32
NUM_STATS = 6
SCALAR_SAVE_BYTES = 512     # RENV_SCALAR_SAVE_BYTES
COUNTER_GAUSSIAN, COUNTER_BAD_ACTION, COUNTER_ORDER_TIMEOUT = 0, 1, 2
TILE_ENVS = {'float32': 1024, 'float64': 512}      # RENV_TILE_ENVS_F32 / _F64
NUM_COUNTERS = 3          # [0] gaussian draws exhausted, [1] invalid actions (include/renv.h)

OK = 0
DR_NONE, DR_UNIFORM, DR_TRUNCNORM, DR_GAUSSIAN, DR_FULLGAUSSIAN = 0, 1, 2, 3, 4
DR_TYPE_IDS = {"uniform": DR_UNIFORM, "truncnorm": DR_TRUNCNORM, "gaussian": DR_GAUSSIAN,
               "fullgaussian": DR_FULLGAUSSIAN}
EULER, SEMI_IMPLICIT = 0, 1


class DrCfg(ctypes.Structure):
    """struct renv_dr_cfg (include/renv.h)."""
    _fields_ = [("dr_type", ctypes.c_int32), ("dim", ctypes.c_int32),
                ("a", ctypes.c_double * MAX_DIM), ("b", ctypes.c_double * MAX_DIM),
                ("lb", ctypes.c_double * MAX_DIM), ("factor", ctypes.c_double * (MAX_DIM * MAX_DIM))]


class CartpoleEnv(ctypes.Structure):
    """struct renv_cartpole_env (include/renv.h)."""
    _fields_ = [("state", ctypes.c_void_p), ("xi", ctypes.c_void_p), ("elapsed", ctypes.c_void_p),
                ("episode", ctypes.c_void_p), ("beyond", ctypes.c_void_p), ("elapsed16", ctypes.c_void_p),
                ("progress", ctypes.c_void_p),
                ("n", ctypes.c_int64), ("ld", ctypes.c_int64),
                ("env_id0", ctypes.c_uint64), ("seed", ctypes.c_uint64)]


class ObsNoise(ctypes.Structure):
    """struct renv_obs_noise (include/renv.h)."""
    _fields_ = [("obs", ctypes.c_void_p), ("std", ctypes.c_double)]


class EpisodeLog(ctypes.Structure):
    """struct renv_episode_log (include/renv.h)."""
    _fields_ = [("xi", ctypes.c_void_p), ("final_state", ctypes.c_void_p), ("length", ctypes.c_void_p),
                ("truncated", ctypes.c_void_p), ("end_tick", ctypes.c_void_p), ("count", ctypes.c_void_p),
                ("capacity", ctypes.c_int64)]


class MlpPolicy(ctypes.Structure):
    """struct renv_mlp_policy (include/renv.h)."""
    _fields_ = [("params", ctypes.c_void_p), ("activation", ctypes.c_int32)]


class Trajectory(ctypes.Structure):
    """struct renv_trajectory (include/renv.h)."""
    _fields_ = [("obs", ctypes.c_void_p), ("action", ctypes.c_void_p), ("done", ctypes.c_void_p),
                ("logp", ctypes.c_void_p), ("truncated", ctypes.c_void_p), ("final_obs", ctypes.c_void_p),
                ("capacity", ctypes.c_int32)]


class Transitions(ctypes.Structure):
    """struct renv_transitions (include/renv.h)."""
    _fields_ = [("obs", ctypes.c_void_p), ("next_obs", ctypes.c_void_p), ("action", ctypes.c_void_p),
                ("window", ctypes.c_void_p), ("T", ctypes.c_int64), ("W", ctypes.c_int32)]


_vp, _i64, _u64, _u32, _int, _dbl = (ctypes.c_void_p, ctypes.c_int64, ctypes.c_uint64, ctypes.c_uint32,
                                     ctypes.c_int, ctypes.c_double)
_flt = ctypes.c_float
_cfg_p, _env_p, _noise_p = ctypes.POINTER(DrCfg), ctypes.POINTER(CartpoleEnv), ctypes.POINTER(ObsNoise)
_log_p = ctypes.POINTER(EpisodeLog)
_mlp_p = ctypes.POINTER(MlpPolicy)
_traj_p = ctypes.POINTER(Trajectory)
_trans_p = ctypes.POINTER(Transitions)

# name -> (restype, argtypes); must list every function declared in include/renv.h
SIGNATURES = {
    "renv_abi_version": (_int, []),
    "renv_strerror": (ctypes.c_char_p, [_int]),
    "renv_dr_sample_f32": (_int, [_vp, _i64, _cfg_p, _u64, _u64, _u32, _vp, _vp]),
    "renv_dr_sample_f64": (_int, [_vp, _i64, _cfg_p, _u64, _u64, _u32, _vp, _vp]),
    "renv_cartpole_reset_f32": (_int, [_env_p, _vp, _u64, _cfg_p, _vp, _vp]),
    "renv_cartpole_reset_f64": (_int, [_env_p, _vp, _u64, _cfg_p, _vp, _vp]),
    "renv_cartpole_step_f32": (_int, [_env_p, _vp, _vp, _vp, _vp, _int, _int, _int, _u64, _cfg_p, _vp, _vp]),
    "renv_cartpole_step_f64": (_int, [_env_p, _vp, _vp, _vp, _vp, _int, _int, _int, _u64, _cfg_p, _vp, _vp]),
    "renv_cartpole_step_lean_f32": (_int, [_env_p, _vp, _vp, _vp, _int, _int, _u64, _cfg_p, _vp, _vp]),
    "renv_cartpole_reset_noisy_f32": (_int, [_env_p, _noise_p, _vp, _u64, _cfg_p, _vp, _vp]),
    "renv_cartpole_reset_noisy_f64": (_int, [_env_p, _noise_p, _vp, _u64, _cfg_p, _vp, _vp]),
    "renv_cartpole_step_noisy_f32": (_int, [_env_p, _noise_p, _vp, _vp, _vp, _vp, _int, _int, _int, _u64, _cfg_p, _vp, _vp]),
    "renv_cartpole_step_noisy_f64": (_int, [_env_p, _noise_p, _vp, _vp, _vp, _vp, _int, _int, _int, _u64, _cfg_p, _vp, _vp]),
    "renv_cartpole_rollout_f32": (_int, [_env_p, ctypes.POINTER(_dbl), _dbl, _int, _int, _int, _u64, _cfg_p, _vp, _vp, _vp]),
    "renv_cartpole_rollout_f64": (_int, [_env_p, ctypes.POINTER(_dbl), _dbl, _int, _int, _int, _u64, _cfg_p, _vp, _vp, _vp]),
    "renv_cartpole_rollout_noisy_f32": (_int, [_env_p, _noise_p, ctypes.POINTER(_dbl), _dbl, _int, _int, _int, _u64, _cfg_p, _vp, _vp, _vp]),
    "renv_cartpole_rollout_noisy_f64": (_int, [_env_p, _noise_p, ctypes.POINTER(_dbl), _dbl, _int, _int, _int, _u64, _cfg_p, _vp, _vp, _vp]),
    "renv_cartpole_step_logged_f32": (_int, [_env_p, _log_p, _vp, _vp, _vp, _vp, _int, _int, _u64, _cfg_p, _vp, _vp]),
    "renv_cartpole_step_logged_f64": (_int, [_env_p, _log_p, _vp, _vp, _vp, _vp, _int, _int, _u64, _cfg_p, _vp, _vp]),
    "renv_cartpole_rollout_logged_f32": (_int, [_env_p, _log_p, ctypes.POINTER(_dbl), _dbl, _int, _int, _int, _u64, _cfg_p, _vp, _vp, _vp]),
    "renv_cartpole_rollout_logged_f64": (_int, [_env_p, _log_p, ctypes.POINTER(_dbl), _dbl, _int, _int, _int, _u64, _cfg_p, _vp, _vp, _vp]),
    "renv_cartpole_policy_actions_mlp_f32": (_int, [_env_p, _mlp_p, _vp, _vp, _vp]),
    "renv_cartpole_rollout_mlp_f32": (_int, [_env_p, _mlp_p, _int, _int, _int, _u64, _cfg_p, _vp, _vp, _vp]),
    "renv_cartpole_rollout_mlp_logged_f32": (_int, [_env_p, _log_p, _mlp_p, _int, _int, _int, _u64, _cfg_p, _vp, _vp, _vp]),
    "renv_cartpole_policy_logp_mlp_f32": (_int, [_env_p, _mlp_p, _int, _u64, _vp, _vp, _vp, _vp]),
    "renv_cartpole_collect_mlp_f32": (_int, [_env_p, _mlp_p, _traj_p, _int, _int, _int, _int, _u64, _cfg_p, _vp, _vp, _vp]),
    "renv_cartpole_collect_mlp_logged_f32": (_int, [_env_p, _log_p, _mlp_p, _traj_p, _int, _int, _int, _int, _u64, _cfg_p,
                                                    _vp, _vp, _vp]),
    "renv_cartpole_gae_mlp_f32": (_int, [_env_p, _mlp_p, _traj_p, _int, _flt, _flt, _vp, _vp, _vp, _vp]),
    "renv_cartpole_population_linear_f32": (_int, [_env_p, _vp, _int, _int, _int, _int, _u64, _cfg_p, _vp, _vp, _vp]),
    "renv_cartpole_population_mlp_f32": (_int, [_env_p, _vp, _int, _int, _int, _int, _int, _u64, _cfg_p, _vp, _vp, _vp]),
    "renv_cartpole_transition_loglik_f64": (_int, [_trans_p, _int, _int, _vp, _int, _int, ctypes.POINTER(_dbl), _vp, _vp,
                                                   _vp]),
    "renv_cartpole_scalar_serve": (_int, [_vp, _vp, _u32, _u64, _vp]),
    "renv_random_actions_u8": (_int, [_vp, _i64, _u64, _u64, _u32, _vp]),
    "renv_pack_flags_u8": (_int, [_vp, _vp, _i64, _vp]),
}


class RenvError(RuntimeError):
    """A C-ABI call returned non-zero (negative: argument contract; positive: cudaError_t)."""

    def __init__(self, fn, code, message):
        super().__init__("%s failed with %d: %s" % (fn, code, message))
        self.code = code


_lib = None


def load():
    """Load the shared library (once) and bind every symbol.  Raises if anything is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.isfile(LIB_PATH):
        raise ImportError(
            "random_envs_b200: %s is missing. Build it with `python -m random_envs_b200.build` "
            "(needs nvcc; sm_100a). There is no CPU fallback." % LIB_PATH)
    lib = ctypes.CDLL(LIB_PATH)
    for name, (restype, argtypes) in SIGNATURES.items():
        try:
            fn = getattr(lib, name)
        except AttributeError as exc:
            raise ImportError("random_envs_b200: symbol %s missing from %s" % (name, LIB_PATH)) from exc
        fn.restype, fn.argtypes = restype, argtypes
    if lib.renv_abi_version() != ABI_VERSION:
        raise ImportError("random_envs_b200: ABI version mismatch (library %d, binding %d); rebuild"
                          % (lib.renv_abi_version(), ABI_VERSION))
    _lib = lib
    return lib


def strerror(code):
    return load().renv_strerror(code).decode()


def call(name, *args):
    """Invoke a C-ABI function and raise RenvError on a non-zero status."""
    rc = getattr(load(), name)(*args)
    if rc != OK:
        raise RenvError(name, rc, strerror(rc))


def make_dr_cfg(dr_type, a, b, lb=None, factor=None):
    """Host image of a DR distribution.  dr_type: str key of set_dr_distribution or None.

    fullgaussian: a = mean (normalised space), b / lb = search-bound lo / hi, factor = (dim, dim) F with F F^T = cov.
    """
    cfg = DrCfg()
    if dr_type is None:
        cfg.dr_type, cfg.dim = DR_NONE, 0
        return cfg
    if dr_type not in DR_TYPE_IDS:
        raise Exception("Unknown dr_type:" + str(dr_type))
    dim = len(a)
    if not 1 <= dim <= MAX_DIM:
        raise ValueError("task_dim %d outside [1, %d]" % (dim, MAX_DIM))
    cfg.dr_type, cfg.dim = DR_TYPE_IDS[dr_type], dim
    for i in range(dim):
        cfg.a[i] = float(a[i])
        cfg.b[i] = float(b[i])
        cfg.lb[i] = float(lb[i]) if lb is not None else 0.0
    if factor is not None:
        for i in range(dim):
            for k in range(dim):
                cfg.factor[i * dim + k] = float(factor[i][k])
    return cfg
