"""In-tree build of librenv_b200.so (hand-written sm_100a kernels + the C ABI of include/renv.h).

    python -m random_envs_b200.build [--force]

nvcc cross-compiles without a GPU.  The .so is git-ignored but travels to the GPU box with the
repo snapshot; cudart is linked statically so the library loads on a CPU-only machine too (symbol
check), it just cannot launch there.
"""
import os
import subprocess
import sys

_HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(_HERE, "csrc")
INCLUDE = os.path.join(os.path.dirname(_HERE), "include")
LIB_PATH = os.path.join(_HERE, "librenv_b200.so")
SOURCES = ["renv_abi.cu"]
HEADERS = ["renv_philox.cuh", "renv_dr.cuh", "renv_cartpole.cuh", "renv_kernels.cuh", "renv_rollout_pair.cuh", "renv_pack.cuh", "renv_fullgauss_tc.cuh", "renv_scalar_server.cuh", "renv_step_body.cuh", "renv_rollout_body.cuh", "renv_mlp_policy.cuh", "renv_mlp_rollout_body.cuh", "renv_mlp_gae.cuh", "renv_transition_loglik.cuh"]

NVCC_FLAGS = [
    "-O3", "-std=c++17",
    "-gencode", "arch=compute_100a,code=sm_100a",
    "-lineinfo",
    "--shared", "-Xcompiler", "-fPIC",
    "-Xptxas", "-v",
    "-cudart", "static",
]


def _nvcc():
    for cand in (os.environ.get("NVCC"), "/usr/local/cuda/bin/nvcc", "nvcc"):
        if cand and (os.path.isabs(cand) and os.path.isfile(cand) or not os.path.isabs(cand)):
            return cand
    return "nvcc"


def is_stale():
    if not os.path.isfile(LIB_PATH):
        return True
    built = os.path.getmtime(LIB_PATH)
    deps = [os.path.join(CSRC, f) for f in SOURCES + HEADERS] + [os.path.join(INCLUDE, "renv.h")]
    return any(os.path.getmtime(d) > built for d in deps)


def build(force=False, verbose=False):
    """Compile the library if missing or older than its sources.  Returns the .so path."""
    if not force and not is_stale():
        return LIB_PATH
    cmd = [_nvcc()] + NVCC_FLAGS + ["-I", INCLUDE, "-o", LIB_PATH] + [os.path.join(CSRC, s) for s in SOURCES]
    proc = subprocess.run(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)
    if verbose or proc.returncode != 0:
        sys.stderr.write(proc.stdout)
    if proc.returncode != 0:
        raise RuntimeError("nvcc failed (%d): %s" % (proc.returncode, " ".join(cmd)))
    with open(os.path.join(_HERE, "librenv_b200.ptxas.log"), "w") as f:
        f.write(proc.stdout)
    return LIB_PATH


if __name__ == "__main__":
    print(build(force="--force" in sys.argv, verbose=True))
