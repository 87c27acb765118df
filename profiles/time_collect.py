"""Fused trajectory collection against the greedy fused rollout and a torch-driven collection loop, in one process.

    python profiles/time_collect.py [--out FILE] [--rounds 3] [--cases 20:256,22:64] [--arms rollout,...]

Cases: 2^20 envs x K = 256 and 2^22 envs x K = 64 (a ~10 GB trajectory buffer each, final_obs included), fp32 envs
with uniform DR, a 4-64-64-2 policy with Tanh and with ReLU (PyTorch default init).  Arms, alternated round by round
on the same env, each timed with CUDA events around its K steps:
    rollout          venv.rollout(policy, num_steps=K)                   greedy, nothing recorded (the baseline)
    collect_sample   venv.collect(policy, K, sample=True, out=buf)      one kernel, every step recorded
    collect_greedy   venv.collect(policy, K, sample=False, out=buf)
    torch_fp32       K x { obs copy; l = net(obs); Categorical(logits=l).sample(); log_prob; step(); done /
                     truncated copies } into preallocated (K, N) buffers, TF32 matmul off.  It records no final_obs
                     (step() with auto-reset does not return it), so it writes less than collect.
    torch_tf32       the same with torch.backends.cuda.matmul.allow_tf32 = True
Reported: best-of-rounds env-steps/s per arm, the spread (max / min - 1) of each arm's rounds, and the ratios.
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
    ap.add_argument("--cases", default="20:256,22:64")
    ap.add_argument("--arms", default="rollout,collect_sample,collect_greedy,torch_fp32,torch_tf32")
    args = ap.parse_args()
    out = dict(gpu_info(), rounds=args.rounds, cases=[])
    for case in args.cases.split(","):
        log2n, K = (int(v) for v in case.split(":"))
        n = 1 << log2n
        for act in (nn.Tanh, nn.ReLU):
            torch.manual_seed(0)
            net = nn.Sequential(nn.Linear(4, 64), act(), nn.Linear(64, 64), act(), nn.Linear(64, 2)).cuda()
            policy = renv.MLPPolicy.from_module(net, "cuda")
            env = make_env(n)
            buf = env.trajectory_buffer(K)
            # the torch arm's preallocated buffers
            t_obs = torch.empty((K, n, 4), device="cuda")
            t_act = torch.empty((K, n), dtype=torch.uint8, device="cuda")
            t_logp = torch.empty((K, n), device="cuda")
            t_done = torch.empty((K, n), dtype=torch.bool, device="cuda")
            t_trunc = torch.empty((K, n), dtype=torch.bool, device="cuda")

            def loop(tf32, steps=K):
                def run():
                    torch.backends.cuda.matmul.allow_tf32 = tf32
                    with torch.no_grad():
                        for k in range(steps):
                            t_obs[k].copy_(env.obs)
                            dist = torch.distributions.Categorical(logits=net(t_obs[k]), validate_args=False)
                            a = dist.sample()
                            t_logp[k].copy_(dist.log_prob(a))
                            t_act[k].copy_(a)
                            _, _, done, info = env.step(t_act[k])
                            t_done[k].copy_(done)
                            t_trunc[k].copy_(info["TimeLimit.truncated"])
                    torch.backends.cuda.matmul.allow_tf32 = False
                return run

            arms = dict(rollout=lambda: env.rollout(policy, 0.0, K),
                        collect_sample=lambda: env.collect(policy, K, sample=True, out=buf),
                        collect_greedy=lambda: env.collect(policy, K, sample=False, out=buf),
                        torch_fp32=loop(False), torch_tf32=loop(True))
            arms = {k: v for k, v in arms.items() if k in args.arms.split(",")}
            env.rollout(policy, 0.0, 5)             # warm-up: module load, cuBLAS algorithm choice
            env.collect(policy, 5, out=buf)
            loop(False, 3)()
            loop(True, 3)()
            times = {k: [] for k in arms}
            for _ in range(args.rounds):
                for k, fn in arms.items():
                    times[k].append(timed(fn))
            rec = dict(num_envs=n, steps=K, activation=act.__name__, seconds=times,
                       trajectory_bytes=sum(v.numel() * v.element_size() for v in
                                            (buf._obs, buf._action, buf._done, buf._truncated, buf._logp, buf._final_obs)))
            for k, ts in times.items():
                rec[k] = dict(env_steps_per_s=n * K / min(ts), spread=max(ts) / min(ts) - 1)
            for k in arms:
                if k != "rollout" and "rollout" in arms:
                    rec[k + "_over_rollout"] = min(times["rollout"]) / min(times[k])
            for k in ("torch_fp32", "torch_tf32"):
                if k in arms and "collect_sample" in arms:
                    rec["collect_sample_over_" + k] = min(times[k]) / min(times["collect_sample"])
            out["cases"].append(rec)
            print(json.dumps(dict((k, v) for k, v in rec.items() if k != "seconds")), flush=True)
            del env, buf, t_obs, t_act, t_logp, t_done, t_trunc
            torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
