"""Population evaluation against today's route and against the single-policy ceiling, in one process.

    python profiles/time_population.py [--out FILE] [--rounds 3] [--steps 500] [--subset 256] [--only linear|mlp]

Cases (fp32, uniform DR, K = 500 env-steps per member and env):
    linear          P x E = 4096 x 256, 65536 x 16, 256 x 4096
    MLP Tanh, ReLU  P x E = 1024 x 128, 256 x 1024, 64 x 16384      (4-64-64-2, PyTorch default init)
Arms, alternated round by round, best of `rounds` with the spread kept:
    population   env.evaluate_population(policies, K) on an env of E envs             (one kernel)
    loop         for each member: env.reset(); env.rollout(policy_p, K) on one env of E envs (2 launches per member);
                 for P > subset the first `subset` members are timed and the time is scaled by P / subset
    ceiling      env.rollout(policy_0, K) on one env of P E envs                     (the single-policy rollout)
env-steps/s = P E K / time.  Times are CUDA events around an arm.  Every member's statistics of the population arm are
checked against the loop arm's for the members the loop ran (they must be equal bit for bit).
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
LINEAR_CASES = [(4096, 256), (65536, 16), (256, 4096)]
MLP_CASES = [(1024, 128), (256, 1024), (64, 16384)]


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
    return env


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / 1e3


def linear_population(P):
    g = torch.Generator().manual_seed(P)
    w = torch.randn((P, 5), generator=g) * torch.tensor([0.5, 0.5, 3.0, 1.0, 0.2]) + torch.tensor([0.0, 0.0, 1.0, 0.5, 0.0])
    return w.float().cuda()


def mlp_population(P, act):
    torch.manual_seed(P)
    nets = [nn.Sequential(nn.Linear(4, 64), act(), nn.Linear(64, 64), act(), nn.Linear(64, 2)) for _ in range(P)]
    return renv.MLPPopulation.from_modules(nets, "cuda")


def run_case(kind, P, E, K, rounds, subset):
    pop = linear_population(P) if kind == "linear" else mlp_population(P, nn.Tanh if kind == "mlp_tanh" else nn.ReLU)
    member = (lambda p: pop.member(p)) if kind != "linear" else (lambda p: pop[p])
    members = [member(p) for p in range(min(P, subset))]
    if kind == "linear":
        rows = [m.double().cpu().tolist() for m in members]
        args = [(r[:4], r[4]) for r in rows]
    else:
        args = [(m, 0.0) for m in members]
    small, big = make_env(E), make_env(P * E)
    tick0 = small._tick
    zero = torch.tensor([0.0, 0.0, 0.0, float("inf"), float("-inf"), 0.0], dtype=torch.float64, device="cuda")
    out = {}

    def population():
        small._tick = tick0
        out["population"] = small.evaluate_population(pop, K)

    def loop():
        rows = []
        for w, b in args:
            small._tick = tick0
            small.stats_tensor.copy_(zero)          # on the device: no host round trip between members
            small.reset()
            small.rollout(w, b, K)
            rows.append(small.stats_tensor.clone())
        out["loop"] = torch.stack(rows)

    def ceiling():
        big.rollout(args[0][0], args[0][1], K)

    arms = dict(population=population, loop=loop, ceiling=ceiling)
    # warm-up: module load, every launch shape of the timed window
    small.evaluate_population(pop, 2)
    small.reset()
    small.rollout(args[0][0], args[0][1], 2)
    big.reset()
    big.rollout(args[0][0], args[0][1], 2)
    times = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            times[k].append(timed(fn))
    equal = bool(torch.equal(out["population"][:len(args)], out["loop"]))
    scale = P / len(args)
    best = {k: min(v) * (scale if k == "loop" else 1.0) for k, v in times.items()}
    rate = {k: P * E * K / t for k, t in best.items()}
    case = dict(kind=kind, P=P, E=E, K=K, loop_members_timed=len(args), seconds=times,
                env_steps_per_s=rate, spread={k: max(v) / min(v) - 1.0 for k, v in times.items()},
                population_over_ceiling=rate["population"] / rate["ceiling"],
                population_over_loop=rate["population"] / rate["loop"], stats_equal_to_loop=equal)
    print(json.dumps(dict((k, v) for k, v in case.items() if k != "seconds")), flush=True)
    del small, big, pop
    torch.cuda.empty_cache()
    return case


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--subset", type=int, default=256)
    ap.add_argument("--only", default=None, choices=("linear", "mlp"))
    args = ap.parse_args()
    info = gpu_info()
    print(json.dumps(info), flush=True)
    out = dict(info, steps=args.steps, rounds=args.rounds, cases=[])
    plan = []
    if args.only in (None, "linear"):
        plan += [("linear", P, E) for P, E in LINEAR_CASES]
    if args.only in (None, "mlp"):
        plan += [(kind, P, E) for kind in ("mlp_tanh", "mlp_relu") for P, E in MLP_CASES]
    for kind, P, E in plan:
        out["cases"].append(run_case(kind, P, E, args.steps, args.rounds, args.subset))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
