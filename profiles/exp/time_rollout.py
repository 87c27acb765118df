"""Timing of the fused-rollout kernels of the built library: python profiles/exp/time_rollout.py
Prints env-steps/s for the three bench policies (survive, reset-heavy, random) plus a fingerprint of the final device
state, so that two builds can be checked against each other (the trajectories must be bit-identical)."""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.join(os.path.dirname(os.path.abspath(__file__)), "..", ".."))

import torch  # noqa: E402

from random_envs_b200.vector_env import RandomCartPoleVecEnv  # noqa: E402


def fingerprint(env):
    b = env._alloc()
    n = env.num_envs
    s = b["state"][:, :n].contiguous().view(torch.int32).to(torch.int64)
    xi = b["xi"][:n].contiguous().view(torch.int32).to(torch.int64)
    return [int(s.sum().item()), int(xi.sum().item()), int(env.elapsed.to(torch.int64).sum().item()),
            int(env.episode.to(torch.int64).sum().item())]


def run(n, K, w, dr, reps, dtype="float32"):
    env = RandomCartPoleVecEnv(n, dtype=dtype, seed=7)
    if dr:
        env.set_dr_distribution("uniform", [9.0, 10.6, 0.8, 1.2, 0.08, 0.12, 0.4, 0.6])
        env.set_dr_training(True)
    env.reset()
    env.rollout(w, 0.0, K)                                  # warm-up (and the fingerprint run)
    stats = env.episode_stats()
    fp = fingerprint(env)
    ms = []
    for _ in range(reps):
        env.seed(7)
        env.reset()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        env.rollout(w, 0.0, K)
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    ms.sort()
    med = ms[len(ms) // 2]
    return {"env_steps_per_s": n * K / (med * 1e-3), "ms": med, "episodes": stats["episodes"],
            "mean_return": stats["mean_return"], "fingerprint": fp}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--log2n", type=int, default=24)
    ap.add_argument("--K", type=int, default=500)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--no-dr", action="store_true")
    ap.add_argument("--only", default="")
    a = ap.parse_args()
    n = 1 << a.log2n
    out = {"n": n, "K": a.K}
    for name, w in (("survive", [0.1, 0.1, 1.0, 0.3]), ("resetheavy", [0.0, 0.0, 1.0, 0.0]), ("random", None)):
        if a.only and name not in a.only.split(","):
            continue
        out[name] = run(n, a.K, w, not a.no_dr, a.reps)
    print(json.dumps(out))


if __name__ == "__main__":
    main()
