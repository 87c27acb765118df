"""Cost of the episode log: logged vs unlogged step() and rollout(), alternated in one process on the same seeded envs.

    python profiles/time_episode_log.py [--out FILE] [--rounds 5]

Cases: fp32 step with random actions and uniform DR (SURVEY cfg 2) on 2^20 envs with tile ordering and on 2^24 envs;
2^24 x 500 fp32 rollouts under w = (0.1, 0.1, 1, 0.3), (0, 0, 1, 0) and the random policy; a 2^23 x 500 fp64 rollout.
Each case builds two envs with the same seed, one with a log (capacity 1) and one without; they evolve identically
(the log perturbs nothing), and their timed blocks alternate.  Times are CUDA events around a block of calls.  Step
actions cycle through 16 pre-drawn random action vectors so that no action kernel runs inside the timed blocks.
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

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


def make_env(n, dtype, tile_ordering, logged):
    env = renv.RandomCartPoleVecEnv(n, dtype=dtype, seed=21, tile_ordering=tile_ordering)
    env.set_dr_distribution("uniform", SEARCH)
    env.set_dr_training(True)
    env.reset()
    if logged:
        env.start_episode_log(1)
    return env


def time_block(fn, reps):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    for _ in range(reps):
        fn()
    end.record()
    end.synchronize()
    return start.elapsed_time(end) / reps * 1e3          # us per call


def run_case(name, arms, reps, rounds, env_steps_per_call):
    for fn in arms.values():                             # warm-up
        time_block(fn, max(2, reps // 4))
    times = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            times[k].append(time_block(fn, reps))
    best = {k: min(v) for k, v in times.items()}
    out = dict(case=name, us_per_call={k: round(v, 2) for k, v in best.items()},
               all_rounds_us={k: [round(x, 2) for x in v] for k, v in times.items()},
               env_steps_per_s={k: "%.3g" % (env_steps_per_call / (v * 1e-6)) for k, v in best.items()},
               logged_over_unlogged=round(best["logged"] / best["unlogged"], 4))
    print(json.dumps(out), flush=True)
    return out


def step_case(n, tile_ordering, reps, rounds):
    envs = dict(unlogged=make_env(n, "float32", tile_ordering, False), logged=make_env(n, "float32", tile_ordering, True))
    actions = []
    pool = envs["unlogged"]
    for _ in range(16):
        actions.append(pool.sample_actions(out=torch.empty(n, dtype=torch.uint8, device="cuda")))
        pool._tick += 1
    for e in envs.values():
        e._tick = 1
    arms = {}
    for k, e in envs.items():
        e.step(actions[0])
        counter = [0]

        def step(e=e, counter=counter):
            counter[0] += 1
            e.step(actions[counter[0] & 15])
        arms[k] = step
    name = "step f32 random actions, uniform DR, 2^%d envs, tile_ordering=%s" % (n.bit_length() - 1, tile_ordering)
    return run_case(name, arms, reps, rounds, n)


def rollout_case(n, dtype, w, K, rounds):
    envs = dict(unlogged=make_env(n, dtype, None, False), logged=make_env(n, dtype, None, True))
    arms = {k: (lambda e=e: e.rollout(w, 0.0, K)) for k, e in envs.items()}
    name = "rollout %s 2^%d x %d, w=%s" % (dtype, n.bit_length() - 1, K, "random" if w is None else list(w))
    return run_case(name, arms, 1, rounds, n * K)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=5)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "needs the GPU"
    torch.cuda.set_device(0)
    rec = dict(gpu_info(), rounds=args.rounds, results=[])
    print(json.dumps({k: v for k, v in rec.items() if k != "results"}), flush=True)
    rec["results"].append(step_case(1 << 20, True, 400, args.rounds))
    rec["results"].append(step_case(1 << 24, None, 60, args.rounds))
    for w in ((0.1, 0.1, 1.0, 0.3), (0.0, 0.0, 1.0, 0.0), None):
        rec["results"].append(rollout_case(1 << 24, "float32", w, 500, args.rounds))
    rec["results"].append(rollout_case(1 << 23, "float64", (0.1, 0.1, 1.0, 0.3), 500, args.rounds))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(rec, f, indent=1)


if __name__ == "__main__":
    main()
