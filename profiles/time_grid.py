"""Evaluation grids against today's route and against the same work without the grid, in one process.

    python profiles/time_grid.py [--out FILE] [--rounds 3] [--steps 500] [--subset 256]

Cases (fp32, K = 500 env-steps per cell and env; MLPs 4-64-64-2 ReLU, PyTorch default init):
    robustness map, MLP      P x C x E = 1 x 4096 x 32     fixed tasks: 64 gravities x 64 pole lengths
    checkpoint sweep, MLP    16 x 8 x 1024                 8 uniform test distributions
    ADR boundaries, MLP      1 x 8 x 1024                  uniform ranges with one dim pinned at lo or hi (lo = hi)
    ARS, linear              1024 x 4 x 16                 4 uniform distributions
Arms, alternated round by round, best of `rounds` with the spread kept:
    grid       env.evaluate_grid(policies, scenarios, K) on an env of E envs                     (one kernel)
    loop       for each scenario: reconfigure the env (set_task, or set_dr_distribution + set_dr_training), then
               env.evaluate_population(policies, K) on it; for C > subset the first `subset` scenarios are timed and
               the time is scaled by C / subset
    ceiling    env.evaluate_population(policies, K) on one env of C E envs under scenario 0      (no grid)
env-steps/s = P C E K / time.  Times are CUDA events around an arm.  The grid's cells are checked against the loop's for
the scenarios the loop ran (they must be equal bit for bit).
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

import numpy as np  # noqa: E402
import torch  # noqa: E402
from torch import nn  # noqa: E402

import random_envs_b200 as renv  # noqa: E402
from time_population import gpu_info, linear_population, timed  # noqa: E402

SEARCH = np.array([2.0, 20.0, 0.5, 3.0, 0.05, 0.3, 0.1, 1.0])
LO, HI = SEARCH[0::2], SEARCH[1::2]
CASES = [("robustness map", "mlp", 1, "tasks", 4096, 32), ("checkpoint sweep", "mlp", 16, "uniform", 8, 1024),
         ("ADR boundaries", "mlp", 1, "boundaries", 8, 1024), ("ARS", "linear", 1024, "uniform", 4, 16)]


def scenario_list(kind, C):
    """C (kind, value) pairs: ("task", (4,) task) or ("uniform", interleaved distr)."""
    if kind == "tasks":
        side = int(round(C ** 0.5))
        return [("task", [g, 1.0, 0.1, l]) for g in np.linspace(2.0, 20.0, side) for l in np.linspace(0.1, 1.0, side)]
    if kind == "boundaries":        # dim d at its lower (even c) or upper (odd c) bound, the others over their ranges
        mid_lo, mid_hi = LO + 0.25 * (HI - LO), HI - 0.25 * (HI - LO)
        out = []
        for c in range(C):
            lo, hi = mid_lo.copy(), mid_hi.copy()
            d = c // 2
            lo[d] = hi[d] = mid_lo[d] if c % 2 == 0 else mid_hi[d]
            out.append(("uniform", np.stack([lo, hi], 1).ravel().tolist()))
        return out
    rng = np.random.default_rng(C)
    out = []
    for _ in range(C):
        lo = LO + (HI - LO) * 0.3 * rng.random(4)
        hi = HI - (HI - LO) * 0.3 * rng.random(4)
        out.append(("uniform", np.stack([lo, hi], 1).ravel().tolist()))
    return out


def scenarios(pairs):
    if all(k == "task" for k, _ in pairs):
        return renv.Scenarios.tasks([v for _, v in pairs], "cuda")
    return renv.Scenarios.distributions("uniform", [v for _, v in pairs], "cuda")


def configure(env, pair):
    kind, value = pair
    if kind == "task":
        env.set_dr_training(False)
        env.set_task(*value)
    else:
        env.set_dr_distribution(kind, value)
        env.set_dr_training(True)


def run_case(name, policy_kind, P, scen_kind, C, E, K, rounds, subset):
    if policy_kind == "linear":
        policies = linear_population(P)
    else:
        torch.manual_seed(P)
        nets = [nn.Sequential(nn.Linear(4, 64), nn.ReLU(), nn.Linear(64, 64), nn.ReLU(), nn.Linear(64, 2)) for _ in range(P)]
        policies = renv.MLPPopulation.from_modules(nets, "cuda")
    pairs = scenario_list(scen_kind, C)
    scen = scenarios(pairs)
    timed_pairs = pairs[:min(C, subset)]
    small = renv.RandomCartPoleVecEnv(E, seed=33)
    loop_env = renv.RandomCartPoleVecEnv(E, seed=33)
    big = renv.RandomCartPoleVecEnv(C * E, seed=33)
    configure(big, pairs[0])
    tick0 = small._tick
    out = {}

    def grid():
        small._tick = tick0
        out["grid"] = small.evaluate_grid(policies, scen, K)

    def loop():
        cols = []
        for pair in timed_pairs:
            configure(loop_env, pair)
            loop_env._tick = tick0
            cols.append(loop_env.evaluate_population(policies, K))
        out["loop"] = torch.stack(cols, 1)

    def ceiling():
        big._tick = tick0
        big.evaluate_population(policies, K)

    arms = dict(grid=grid, loop=loop, ceiling=ceiling)
    small.evaluate_grid(policies, scen, 2)          # warm-up: module load, every launch shape of the timed window
    configure(loop_env, pairs[0])
    loop_env.evaluate_population(policies, 2)
    big.evaluate_population(policies, 2)
    times = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            times[k].append(timed(fn))
    for e in (small, loop_env, big):
        e.check_dr_violations()
    equal = bool(torch.equal(out["grid"][:, :len(timed_pairs)], out["loop"]))
    scale = C / len(timed_pairs)
    best = {k: min(v) * (scale if k == "loop" else 1.0) for k, v in times.items()}
    rate = {k: P * C * E * K / t for k, t in best.items()}
    case = dict(case=name, policies=policy_kind, P=P, C=C, E=E, K=K, loop_scenarios_timed=len(timed_pairs),
                seconds=times, best_seconds=best, env_steps_per_s=rate,
                spread={k: max(v) / min(v) - 1.0 for k, v in times.items()},
                grid_over_ceiling=rate["grid"] / rate["ceiling"], grid_over_loop=rate["grid"] / rate["loop"],
                cells_equal_to_loop=equal)
    print(json.dumps(dict((k, v) for k, v in case.items() if k != "seconds")), flush=True)
    del small, loop_env, big, policies
    torch.cuda.empty_cache()
    return case


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--subset", type=int, default=256)
    args = ap.parse_args()
    info = gpu_info()
    print(json.dumps(info), flush=True)
    out = dict(info, steps=args.steps, rounds=args.rounds, cases=[])
    for case in CASES:
        out["cases"].append(run_case(*case, args.steps, args.rounds, args.subset))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
