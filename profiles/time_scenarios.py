"""Per-env task scenarios in the training path against the same work without them, in one process.

    python profiles/time_scenarios.py [--out FILE] [--rounds 3] [--quick]

Cases (fp32; B200 card name and power limit are read in the same run):
    step        the lean 54-byte step at 2^20 and 2^24 envs under fixed random actions (an episode ends every ~10
                steps) and under the linear policy a = [theta > 0] (one elementwise kernel per step writes the env's
                action buffer; every arm runs it).  200 timed steps after 20 warm-up steps.  Three arms:
                  plain    one uniform DR config over the search box;
                  scen     the 9 ADR-boundary rows of that box (Scenarios.adr_boundaries), half the envs on row 0 (the
                           box), the other half spread over the 8 boundary rows.  Its boundary envs run other tasks
                           (a pole pinned at its shortest length falls sooner), so it also does other work;
                  scen_box the same assignment on 9 copies of the box row: the plain arm's work exactly, through the
                           scenario kernels -- the cost of the mechanism alone.
    mlp         collect (sampled) and rollout under a 4-64-64-2 ReLU MLP at 2^17 envs, K = 256 and 500, same arms.
    linear      rollout of a linear policy at 2^20 envs, K = 500: plain (the FFMA2 pair kernel) vs the scen arms (the
                generic one-env-per-thread body); and the random policy (every arm on the generic body).
    workaround  one scen collect on N envs (9 ADR rows, N / 9 envs each) vs 9 env objects of N / 9 envs, each with its
                own uniform config and its own collect, at N = 2^16 and 2^20 (ReLU MLP, K = 256).
Arms alternate round by round; the best of `rounds` is reported with the spread (max / min - 1).  Times are CUDA events
around an arm.  Outputs are checked at the timed sizes: the envs of row 0 (the box itself) must equal the plain env's
envs bit for bit (state, xi, elapsed, episode counters, trajectory rows), every env of scen_box must equal the plain
env's, and the workaround's env objects must equal the scen env's envs of their row.
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
from time_population import gpu_info, timed  # noqa: E402

SEARCH = np.array([2.0, 20.0, 0.5, 3.0, 0.05, 0.3, 0.1, 1.0])
LO, HI = SEARCH[0::2], SEARCH[1::2]
SEED = 33


def boundary_assignment(n):
    """Half the envs on row 0 (the box), the other half over the 8 boundary rows."""
    i = torch.arange(n, device="cuda")
    return torch.where(i % 2 == 0, torch.zeros_like(i), 1 + (i // 2) % 8)


ARMS = ("plain", "scen", "scen_box")


def make_env(n, arm, **kw):
    env = renv.RandomCartPoleVecEnv(n, seed=SEED, **kw)
    env.set_dr_distribution("uniform", SEARCH)
    env.set_dr_training(True)
    if arm == "scen":
        env.set_scenarios(renv.Scenarios.adr_boundaries(LO, HI, device="cuda"), boundary_assignment(n))
    elif arm == "scen_box":
        box = renv.Scenarios.distributions("uniform", [SEARCH.tolist()], device="cuda")
        env.set_scenarios(renv.Scenarios.cat(*[box] * 9), boundary_assignment(n))
    return env


def ratios(res):
    """scen / plain and scen_box / plain as speeds (plain time over arm time)."""
    res["ratio_scen_over_plain"] = res["plain"]["best_s"] / res["scen"]["best_s"]
    res["ratio_scen_box_over_plain"] = res["plain"]["best_s"] / res["scen_box"]["best_s"]


def check(envs, n, bufs=None, fields=("obs", "actions", "logp", "dones")):
    """row 0 of scen and every env of scen_box equal plain, bit for bit."""
    row0 = boundary_assignment(n) == 0
    every = torch.ones(n, dtype=torch.bool, device="cuda")
    p = snap(envs["plain"])
    ok = equal_on(p, snap(envs["scen"]), row0) and equal_on(p, snap(envs["scen_box"]), every)
    for f in fields if bufs else ():
        ok = ok and torch.equal(getattr(bufs["plain"], f)[:, row0], getattr(bufs["scen"], f)[:, row0])
        ok = ok and torch.equal(getattr(bufs["plain"], f), getattr(bufs["scen_box"], f))
    for e in envs.values():
        e.check_dr_violations()
    return bool(ok)


def mlp(seed=0):
    torch.manual_seed(seed)
    return renv.MLPPolicy.from_module(nn.Sequential(nn.Linear(4, 64), nn.ReLU(), nn.Linear(64, 64), nn.ReLU(),
                                                    nn.Linear(64, 2)), "cuda")


def snap(env, rows=None):
    s = dict(state=env.state, xi=env.get_task(), elapsed=env.elapsed, episode=env.episode)
    return {k: (v[rows] if rows is not None else v).clone() for k, v in s.items()}


def equal_on(a, b, rows):
    return all(torch.equal(a[k][rows], b[k][rows]) for k in a)


def alternate(arms, rounds):
    """{name: [seconds per round]} of callables run alternately."""
    times = {k: [] for k in arms}
    for _ in range(rounds):
        for k, fn in arms.items():
            times[k].append(timed(fn))
    return times


def summary(times, work):
    out = {}
    for k, ts in times.items():
        best = min(ts)
        out[k] = dict(best_s=best, spread=max(ts) / best - 1.0, rate=work / best, rounds_s=ts)
    return out


def case_step(n, policy, rounds, steps=200, warm=20):
    envs = {k: make_env(n, k, max_episode_steps=500, lean=True) for k in ARMS}
    g = torch.Generator(device="cuda").manual_seed(1)
    fixed = torch.randint(0, 2, (n,), generator=g, device="cuda", dtype=torch.uint8)

    def runner(env):
        b = env._alloc()
        own = env._own_action_view()
        theta = b["state"][2, :n]
        if policy == "random":
            own.copy_(fixed)

        def run(k=steps):
            for _ in range(k):
                if policy == "linear":
                    torch.gt(theta, 0, out=own.view(torch.bool))
                env.step(own)
        return run
    runs = {k: runner(e) for k, e in envs.items()}
    for e in envs.values():
        e.reset()
    for r in runs.values():
        r(warm)
    torch.cuda.synchronize()
    times = alternate(runs, rounds)
    res = summary(times, n * steps)
    ratios(res)
    res["outputs_equal"] = check(envs, n)
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
    for r in runs.values():
        r()
    times = alternate(runs, rounds)
    res = summary(times, n * K)
    ratios(res)
    res["outputs_equal"] = check(envs, n, bufs if what == "collect" else None)
    return res


def case_linear(n, K, rounds):
    envs = {k: make_env(n, k, max_episode_steps=500) for k in ARMS}
    for e in envs.values():
        e.reset()
    out = {}
    for policy, w in (("linear", (0.0, 0.2, 1.5, 0.3)), ("random", None)):
        runs = {k: (lambda e=e: e.rollout(w, 0.0, K)) for k, e in envs.items()}
        for r in runs.values():
            r()
        times = alternate(runs, rounds)
        res = summary(times, n * K)
        ratios(res)
        res["outputs_equal"] = check(envs, n)
        out[policy] = res
    return out


def case_workaround(n, K, rounds):
    C = 9
    m = n // C
    n = m * C
    rows = renv.Scenarios.adr_boundaries(LO, HI, device="cuda")
    scen = renv.RandomCartPoleVecEnv(n, seed=SEED, max_episode_steps=500)
    assign = torch.arange(n, device="cuda") // m          # contiguous blocks: env object c holds the ids of row c
    scen.set_scenarios(rows, assign)
    split = []
    lo, hi = LO, HI
    boxes = [(lo, hi)]
    for k in range(4):
        for v in (lo[k], hi[k]):
            pl, ph = lo.copy(), hi.copy()
            pl[k] = ph[k] = v
            boxes.append((pl, ph))
    for c, (pl, ph) in enumerate(boxes):
        e = renv.RandomCartPoleVecEnv(m, seed=SEED, env_id0=c * m, max_episode_steps=500)
        e.set_dr_distribution("uniform", np.stack([pl, ph], 1).ravel().tolist())
        e.set_dr_training(True)
        split.append(e)
    policy = mlp(2)
    buf = scen.trajectory_buffer(K)
    bufs = [e.trajectory_buffer(K) for e in split]
    for e in [scen] + split:
        e.reset()

    def one():
        scen.collect(policy, K, out=buf)

    def many():
        for e, b in zip(split, bufs):
            e.collect(policy, K, out=b)
    runs = {"scen": one, "nine_envs": many}
    for r in runs.values():
        r()
    times = alternate(runs, rounds)
    res = summary(times, n * K)
    res["speedup_scen_over_nine_envs"] = res["nine_envs"]["best_s"] / res["scen"]["best_s"]
    got = snap(scen)
    ok = True
    for c, e in enumerate(split):
        w = snap(e)
        ok = ok and all(torch.equal(got[k][c * m:(c + 1) * m], w[k]) for k in w)
        ok = ok and torch.equal(buf.obs[:, c * m:(c + 1) * m], bufs[c].obs)
    res["outputs_equal"] = bool(ok)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--quick", action="store_true", help="small sizes: a rehearsal of the script, not a measurement")
    args = ap.parse_args()
    renv.load_library()
    result = dict(info=gpu_info(), rounds=args.rounds, cases=[])
    big = [1 << 14] if args.quick else [1 << 20, 1 << 24]
    for n in big:
        for policy in ("random", "linear"):
            r = case_step(n, policy, args.rounds)
            result["cases"].append(dict(case="step lean", envs=n, policy=policy, **r))
            print(json.dumps(dict(case="step lean", envs=n, policy=policy, ratio=r["ratio_scen_over_plain"],
                                  ratio_box=r["ratio_scen_box_over_plain"], equal=r["outputs_equal"])), flush=True)
    for what in ("collect", "rollout_mlp"):
        for K in ((16,) if args.quick else (256, 500)):
            r = case_mlp(1 << (12 if args.quick else 17), "collect" if what == "collect" else "rollout", K, args.rounds)
            result["cases"].append(dict(case=what, envs=1 << (12 if args.quick else 17), K=K, **r))
            print(json.dumps(dict(case=what, K=K, ratio=r["ratio_scen_over_plain"], ratio_box=r["ratio_scen_box_over_plain"],
                                  equal=r["outputs_equal"])), flush=True)
    n = 1 << (12 if args.quick else 20)
    K = 16 if args.quick else 500
    for policy, r in case_linear(n, K, args.rounds).items():
        result["cases"].append(dict(case="rollout " + policy, envs=n, K=K, **r))
        print(json.dumps(dict(case="rollout " + policy, ratio=r["ratio_scen_over_plain"],
                              ratio_box=r["ratio_scen_box_over_plain"], equal=r["outputs_equal"])), flush=True)
    for n in ((1 << 12,) if args.quick else (1 << 16, 1 << 20)):
        r = case_workaround(n, 16 if args.quick else 256, args.rounds)
        result["cases"].append(dict(case="workaround: 1 scen collect vs 9 env objects", envs=n, **r))
        print(json.dumps(dict(case="workaround", envs=n, speedup=r["speedup_scen_over_nine_envs"],
                              equal=r["outputs_equal"])), flush=True)
    result["all_outputs_equal"] = all(c["outputs_equal"] for c in result["cases"])
    text = json.dumps(result, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print("all outputs equal: %s" % result["all_outputs_equal"])


if __name__ == "__main__":
    main()
