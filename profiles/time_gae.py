"""Fused advantage estimation (gae) against the greedy MLP rollout, a torch GAE and collect alone, in one process.

    python profiles/time_gae.py [--out FILE] [--rounds 3] [--cases 20:256,22:64] [--arms gae,rollout,...]

Cases: 2^20 envs x K = 256 and 2^22 envs x K = 64 (a ~10 GB trajectory buffer with final_obs, plus 3 GB of values,
advantages and returns), fp32 envs with uniform DR and TimeLimit 500, a 4-64-64-2 policy and a 4-64-64-1 critic with
the same activation, Tanh and ReLU (PyTorch default init).  The trajectory is that of a sampled collect.  Arms,
alternated round by round, each timed with CUDA events:
    gae              venv.gae(traj, critic)                       one kernel over the K x N trajectory
    rollout          venv.rollout(policy, num_steps=K)            greedy, nothing recorded: the reference point of
                                                                  DESIGN section 4.9
    torch_tf32       what a PPO implementation runs on the same trajectory: critic(obs) in chunks of 2^22 rows with TF32
                     matmuls, critic(final_obs) where truncated, critic(s_K), then the reverse GAE loop over K
    collect          venv.collect(policy, K, sample=True, out=buf)
    collect_gae      the same followed by venv.gae(buf, critic): one training iteration's data
gae and torch_tf32 run on one env (its clock stays where its collect left it); rollout, collect and collect_gae on a
second env with the same seed.  Both work on sizes far above the 126 MB L2.  Reported: best-of-rounds env-steps/s per
arm, the spread (max / min - 1) of each arm's rounds, and the ratios.
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
CHUNK = 1 << 22
GAMMA, LAM = 0.99, 0.95


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


def torch_gae(env, traj, critic_net, out):
    """The torch path: chunked critic with TF32 matmuls, the truncation bootstrap, the reverse GAE loop."""
    values, adv = out
    K, n = traj.num_steps, traj.num_envs
    torch.backends.cuda.matmul.allow_tf32 = True
    with torch.no_grad():
        obs = traj.obs.reshape(K * n, 4)
        flat = values.view(-1)
        for s in range(0, K * n, CHUNK):
            flat[s:s + CHUNK] = critic_net(obs[s:s + CHUNK]).squeeze(-1)
        trunc, done = traj.truncated, traj.dones
        v_final = torch.zeros_like(values)
        v_final[trunc] = critic_net(traj.final_obs[trunc]).squeeze(-1)
        v_next = critic_net(env.obs).squeeze(-1)
        a = torch.zeros(n, device=values.device)
        for k in range(K - 1, -1, -1):
            nv = torch.where(done[k], v_final[k], v_next)
            delta = 1.0 + GAMMA * nv - values[k]
            a = delta + (GAMMA * LAM) * (~done[k]) * a
            adv[k] = a
            v_next = values[k]
        returns = adv + values
    torch.backends.cuda.matmul.allow_tf32 = False
    return returns


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--cases", default="20:256,22:64")
    ap.add_argument("--arms", default="gae,rollout,torch_tf32,collect,collect_gae")
    args = ap.parse_args()
    out = dict(gpu_info(), rounds=args.rounds, cases=[])
    for case in args.cases.split(","):
        log2n, K = (int(v) for v in case.split(":"))
        n = 1 << log2n
        for act in (nn.Tanh, nn.ReLU):
            torch.manual_seed(0)
            net = nn.Sequential(nn.Linear(4, 64), act(), nn.Linear(64, 64), act(), nn.Linear(64, 2)).cuda()
            critic_net = nn.Sequential(nn.Linear(4, 64), act(), nn.Linear(64, 64), act(), nn.Linear(64, 1)).cuda()
            policy = renv.MLPPolicy.from_module(net, "cuda")
            critic = renv.MLPPolicy.from_module(critic_net, "cuda")
            env, other = make_env(n), make_env(n)
            traj = env.collect(policy, K, sample=True, out=env.trajectory_buffer(K))
            buf = other.trajectory_buffer(K)
            t_out = (torch.empty((K, n), device="cuda"), torch.empty((K, n), device="cuda"))

            def collect_gae():
                other.collect(policy, K, sample=True, out=buf)
                other.gae(buf, critic)

            arms = dict(gae=lambda: env.gae(traj, critic, GAMMA, LAM),
                        rollout=lambda: other.rollout(policy, 0.0, K),
                        torch_tf32=lambda: torch_gae(env, traj, critic_net, t_out),
                        collect=lambda: other.collect(policy, K, sample=True, out=buf),
                        collect_gae=collect_gae)
            arms = {k: v for k, v in arms.items() if k in args.arms.split(",")}
            for fn in arms.values():                # warm-up: module load, cuBLAS algorithm choice, allocator
                fn()
            torch.cuda.synchronize()
            # the torch arm computes what the kernel computes: agreement at the timed size
            env.gae(traj, critic, GAMMA, LAM)
            t_ret = torch_gae(env, traj, critic_net, t_out)
            check = dict(max_abs_value_diff=float((t_out[0] - traj.values).abs().max()),
                         max_abs_advantage_diff=float((t_out[1] - traj.advantages).abs().max()),
                         max_abs_return_diff=float((t_ret - traj.returns).abs().max()),
                         max_abs_advantage=float(traj.advantages.abs().max()),
                         truncated_fraction=float(traj.truncated.float().mean()),
                         done_fraction=float(traj.dones.float().mean()))
            del t_ret
            times = {k: [] for k in arms}
            for _ in range(args.rounds):
                for k, fn in arms.items():
                    times[k].append(timed(fn))
            rec = dict(num_envs=n, steps=K, activation=act.__name__, seconds=times, torch_check=check)
            for k, ts in times.items():
                rec[k] = dict(env_steps_per_s=n * K / min(ts), spread=max(ts) / min(ts) - 1)
            if "gae" in arms and "rollout" in arms:
                rec["gae_over_rollout"] = min(times["rollout"]) / min(times["gae"])
            if "gae" in arms and "torch_tf32" in arms:
                rec["gae_over_torch_tf32"] = min(times["torch_tf32"]) / min(times["gae"])
            if "collect" in arms and "collect_gae" in arms:
                rec["collect_gae_over_collect"] = min(times["collect_gae"]) / min(times["collect"])
            out["cases"].append(rec)
            print(json.dumps(dict((k, v) for k, v in rec.items() if k != "seconds")), flush=True)
            del env, other, traj, buf, t_out
            torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
