"""Fused MLP-policy rollout against a torch-driven loop: the same policy, the same seeded envs, in one process.

    python profiles/time_mlp_rollout.py [--out FILE] [--rounds 3] [--steps 500] [--sizes 20,24] [--arms fused,...]

Cases: 2^20 and 2^24 fp32 envs with uniform DR, 500 env-steps, a 4-64-64-2 policy with Tanh and with ReLU (PyTorch
default init).  Arms, alternated round by round:
    fused        venv.rollout(policy, num_steps=K)                       (one kernel)
    torch_fp32   K x { venv.step(net(venv.obs).argmax(1)) }, torch TF32 matmul off
    torch_tf32   the same with torch.backends.cuda.matmul.allow_tf32 = True
Times are CUDA events around the K steps of an arm.  Algorithmic FLOPs per env-step: 2 (4*64 + 64*64 + 64*2) = 8,960,
plus 128 activations (not counted as FLOPs).
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402
from torch import nn  # noqa: E402

import random_envs_b200 as renv  # noqa: E402

SEARCH = [2.0, 20.0, 0.5, 3.0, 0.05, 0.3, 0.1, 1.0]
FLOPS_PER_STEP = 2 * (4 * 64 + 64 * 64 + 64 * 2)


def gpu_info():
    info = dict(gpu=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        info["power_limit_and_max_sm_clock"] = q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError) as exc:
        info["power_limit_and_max_sm_clock"] = "unknown (%s)" % exc
    return info


def make_env(n):
    env = renv.RandomCartPoleVecEnv(n, seed=33)
    env.set_dr_distribution("uniform", SEARCH)
    env.set_dr_training(True)
    env.reset()
    return env


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--sizes", default="20,24")
    ap.add_argument("--arms", default="fused,torch_fp32,torch_tf32")
    args = ap.parse_args()
    K = args.steps
    out = dict(gpu_info(), steps=K, flops_per_env_step=FLOPS_PER_STEP, cases=[])
    for log2n in [int(v) for v in args.sizes.split(",")]:
        n = 1 << log2n
        for act in (nn.Tanh, nn.ReLU):
            torch.manual_seed(0)
            net = nn.Sequential(nn.Linear(4, 64), act(), nn.Linear(64, 64), act(), nn.Linear(64, 2)).cuda()
            policy = renv.MLPPolicy.from_module(net, "cuda")
            env = make_env(n)

            def fused():
                env.rollout(policy, 0.0, K)

            def loop(tf32):
                def run():
                    torch.backends.cuda.matmul.allow_tf32 = tf32
                    with torch.no_grad():
                        for _ in range(K):
                            env.step(net(env.obs).argmax(1).to(torch.uint8))
                    torch.backends.cuda.matmul.allow_tf32 = False
                return run

            arms = dict(fused=fused, torch_fp32=loop(False), torch_tf32=loop(True))
            arms = {k: v for k, v in arms.items() if k in args.arms.split(",")}
            env.rollout(policy, 0.0, 5)          # warm-up: module load, cuBLAS algorithm choice
            with torch.no_grad():
                for _ in range(3):
                    env.step(net(env.obs).argmax(1).to(torch.uint8))
            times = {k: [] for k in arms}
            for _ in range(args.rounds):
                for k, fn in arms.items():
                    times[k].append(timed(fn))
            case = dict(num_envs=n, activation=act.__name__, seconds=times)
            for k, ts in times.items():
                best = min(ts)
                case[k] = dict(env_steps_per_s=n * K / best, algorithmic_flop_per_s=n * K * FLOPS_PER_STEP / best)
            for k in ("torch_fp32", "torch_tf32"):
                if k in times and "fused" in times:
                    case["fused_over_" + k] = min(times[k]) / min(times["fused"])
            out["cases"].append(case)
            print(json.dumps(dict((k, v) for k, v in case.items() if k != "seconds")), flush=True)
            del env
            torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
