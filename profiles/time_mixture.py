"""Scenario mixtures in the training path against the same work without them, in one process.

    python profiles/time_mixture.py [--out FILE] [--rounds 3] [--quick]

Arms (fp32; B200 card name, power limit and max SM clock are read in the same run):
    mix9      set_scenario_mixture over the 9 ADR rows of the search box (Scenarios.adr_boundaries), weights
              [1 - p_b] + [p_b / 8] * 8 with p_b = 0.5: other tasks than the box, so other work as well;
    mix_box   the mixture over 9 copies of the box row: the work of scen_box and plain exactly, through the mixture
              kernels (a draw, a table load and a row load per reset, statistics per row);
    scen_box  set_scenarios on the same 9 box rows;
    plain     one uniform DR config over the box (the plain kernels);
    resample  today's route to per-iteration resampling: torch.multinomial assignment, set_scenarios, collect.
Cases: the lean step at 2^20 and 2^24 envs under fixed random actions (200 timed steps); ReLU MLP collect and rollout
at 2^17 envs, K = 256 and 500; the random-policy rollout at 2^20, K = 500; an empirical task set of C = 4096 fixed
tasks with uniform weights (collect, 2^17 envs, K = 256; global statistics path) against set_scenarios on a random
assignment of the same rows.  Arms alternate round by round; the best of `rounds` is reported with the spread.  Times
are CUDA events around an arm.  Outputs are checked at the timed sizes: mix_box, scen_box and plain envs equal bit for
bit (state, xi, elapsed, episode counters, trajectory rows).  mix9, resample and the empirical set run other tasks and
have no twin: their outputs are not checked here (outputs_equal null, outputs_unchecked).
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

import random_envs_b200 as renv  # noqa: E402
from time_population import gpu_info, timed  # noqa: E402
from time_scenarios import LO, HI, SEARCH, SEED, alternate, equal_on, mlp, snap, summary  # noqa: E402

P_B = 0.5
ADR_WEIGHTS = [1.0 - P_B] + [P_B / 8] * 8
ARMS = ("plain", "scen_box", "mix_box", "mix9")


def box9():
    box = renv.Scenarios.distributions("uniform", [SEARCH.tolist()], device="cuda")
    return renv.Scenarios.cat(*[box] * 9)


def make_env(n, arm, **kw):
    env = renv.RandomCartPoleVecEnv(n, seed=SEED, **kw)
    env.set_dr_distribution("uniform", SEARCH)
    env.set_dr_training(True)
    if arm == "scen_box":
        env.set_scenarios(box9(), torch.arange(n, device="cuda") % 9)
    elif arm == "mix_box":
        env.set_scenario_mixture(box9(), ADR_WEIGHTS)
    elif arm == "mix9":
        env.set_scenario_mixture(renv.Scenarios.adr_boundaries(LO, HI, device="cuda"), ADR_WEIGHTS)
    env.reset()
    return env


def ratios(res):
    p = res["plain"]["best_s"]
    for k in ("scen_box", "mix_box", "mix9"):
        res["ratio_%s_over_plain" % k] = p / res[k]["best_s"]
    res["ratio_mix_box_over_scen_box"] = res["scen_box"]["best_s"] / res["mix_box"]["best_s"]


def check(envs, n, bufs=None, fields=("obs", "actions", "logp", "dones")):
    every = torch.ones(n, dtype=torch.bool, device="cuda")
    p = snap(envs["plain"])
    ok = equal_on(p, snap(envs["scen_box"]), every) and equal_on(p, snap(envs["mix_box"]), every)
    for f in fields if bufs else ():
        ok = ok and torch.equal(getattr(bufs["plain"], f), getattr(bufs["scen_box"], f))
        ok = ok and torch.equal(getattr(bufs["plain"], f), getattr(bufs["mix_box"], f))
    for e in envs.values():
        e.check_dr_violations()
    return bool(ok)


def case_step(n, rounds, steps=200, warm=20):
    envs = {k: make_env(n, k, max_episode_steps=500, lean=True) for k in ARMS}
    g = torch.Generator(device="cuda").manual_seed(1)
    fixed = torch.randint(0, 2, (n,), generator=g, device="cuda", dtype=torch.uint8)

    def runner(env):
        own = env._own_action_view()
        own.copy_(fixed)

        def run(k=steps):
            for _ in range(k):
                env.step(own)
        return run
    runs = {k: runner(e) for k, e in envs.items()}
    for e in envs.values():
        e.reset()
    for r in runs.values():
        r(warm)
    torch.cuda.synchronize()
    res = summary(alternate(runs, rounds), n * steps)
    ratios(res)
    res["outputs_equal"] = check(envs, n)
    res["outputs_unchecked"] = ["mix9"]
    return res


def case_mlp(n, what, K, rounds):
    envs = {k: make_env(n, k, max_episode_steps=500) for k in ARMS}
    policy = mlp(1)
    bufs = {k: e.trajectory_buffer(K) for k, e in envs.items()}
    for e in envs.values():
        e.reset()

    def runner(k):
        e = envs[k]
        return (lambda: e.collect(policy, K, out=bufs[k])) if what == "collect" else (lambda: e.rollout(policy, 0.0, K))
    runs = {k: runner(k) for k in envs}
    if what == "collect":       # (e): a new assignment drawn from the weights, set_scenarios, then collect
        rs = make_env(n, "plain", max_episode_steps=500)
        rs.reset()
        rows9 = renv.Scenarios.adr_boundaries(LO, HI, device="cuda")
        wt = torch.tensor(ADR_WEIGHTS, device="cuda")
        rbuf = rs.trajectory_buffer(K)

        def resample():
            rs.set_scenarios(rows9, torch.multinomial(wt, n, replacement=True))
            rs.collect(policy, K, out=rbuf)
        runs["resample"] = resample
    for r in runs.values():
        r()
    res = summary(alternate(runs, rounds), n * K)
    ratios(res)
    if "resample" in res:
        res["ratio_mix9_over_resample"] = res["resample"]["best_s"] / res["mix9"]["best_s"]
    res["outputs_equal"] = check(envs, n, bufs if what == "collect" else None)
    res["outputs_unchecked"] = ["mix9"] + (["resample"] if "resample" in res else [])     # no twin: other tasks
    return res


def case_random_rollout(n, K, rounds):
    envs = {k: make_env(n, k, max_episode_steps=500) for k in ARMS}
    for e in envs.values():
        e.reset()
    runs = {k: (lambda e=e: e.rollout(None, 0.0, K)) for k, e in envs.items()}
    for r in runs.values():
        r()
    res = summary(alternate(runs, rounds), n * K)
    ratios(res)
    res["outputs_equal"] = check(envs, n)
    res["outputs_unchecked"] = ["mix9"]
    return res


def case_empirical(n, K, rounds, C=4096):
    rng = np.random.default_rng(5)
    tasks = rng.uniform(LO, HI, size=(C, 4))
    rows = renv.Scenarios.tasks(tasks, "cuda")
    mix = renv.RandomCartPoleVecEnv(n, seed=SEED, max_episode_steps=500)
    mix.set_scenario_mixture(rows, np.ones(C))
    scen = renv.RandomCartPoleVecEnv(n, seed=SEED, max_episode_steps=500)
    scen.set_scenarios(rows, torch.from_numpy(rng.integers(0, C, n)).cuda())
    policy = mlp(3)
    bufs = {k: e.trajectory_buffer(K) for k, e in (("mix", mix), ("scen", scen))}
    for e in (mix, scen):
        e.reset()
    runs = {"mix": lambda: mix.collect(policy, K, out=bufs["mix"]), "scen": lambda: scen.collect(policy, K, out=bufs["scen"])}
    for r in runs.values():
        r()
    res = summary(alternate(runs, rounds), n * K)
    res["ratio_mix_over_scen"] = res["scen"]["best_s"] / res["mix"]["best_s"]
    res["outputs_equal"] = None         # no twin: the arms run different tasks (the GPU tests cover the C > 64 path)
    for e in (mix, scen):
        e.check_dr_violations()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--quick", action="store_true", help="small sizes: a rehearsal of the script, not a measurement")
    args = ap.parse_args()
    renv.load_library()
    result = dict(info=gpu_info(), rounds=args.rounds, cases=[])

    def report(case, **r):
        result["cases"].append(dict(case=case, **r))
        print(json.dumps({k: v for k, v in r.items() if k.startswith(("ratio", "envs", "K", "outputs"))} | dict(case=case)),
              flush=True)
    for n in ([1 << 14] if args.quick else [1 << 20, 1 << 24]):
        report("step lean, random actions", envs=n, **case_step(n, args.rounds))
    n = 1 << (12 if args.quick else 17)
    for what in ("collect", "rollout_mlp"):
        for K in ((16,) if args.quick else (256, 500)):
            report(what, envs=n, K=K, **case_mlp(n, "collect" if what == "collect" else "rollout", K, args.rounds))
    n, K = (1 << 12, 16) if args.quick else (1 << 20, 500)
    report("rollout random", envs=n, K=K, **case_random_rollout(n, K, args.rounds))
    n, K = (1 << 12, 16) if args.quick else (1 << 17, 256)
    report("empirical task set C=4096, collect", envs=n, K=K, **case_empirical(n, K, args.rounds))
    # over the arms with a twin (plain, scen_box, mix_box); mix9, resample and the empirical set have none
    result["all_outputs_equal"] = all(c["outputs_equal"] for c in result["cases"] if c["outputs_equal"] is not None)
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print("all outputs equal: %s" % result["all_outputs_equal"])


if __name__ == "__main__":
    main()
