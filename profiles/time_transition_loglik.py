"""Offline DR log-likelihood (TransitionDataset.log_likelihood) against a torch float64 arm and the fp64 fused rollout.

    python profiles/time_transition_loglik.py [--out FILE] [--rounds 3] [--torch-cases C:M:lam,...]

Data: W = 8192 windows of noisy fp64 cart-pole transitions (RandomCartPoleVecEnv(noisy=True, dtype="float64") under
sample_actions() at xi* = (12, 1.5, 0.2, 0.7), noise_level 1e-4), candidates drawn truncnorm around xi* (std 2 % of
the mean), eps = 2e-4.  Cases: C in {16, 64} x M in {256, 1024} x lam in {1, 5} with Euler, and C = 64, M = 1024,
lam = 1 semi-implicit.  Arms, alternated round by round, each timed with CUDA events (best of rounds, with the spread
max / min - 1):
    kernel   data.log_likelihood(xi, lam)                         the two launches of renv_cartpole_transition_loglik_f64
    torch    the same objective in torch float64: dynamics vectorised over (windows, samples) in chunks, then mean,
             covariance, Cholesky and log-density per window -- run on --torch-cases, checked against the kernel
    rollout  the fp64 fused rollout, 2^24 envs x 500 steps, uniform DR, w = (0.1, 0.1, 1, 0.3) (bench.py's
             rollout_f64_survive): the reference rate of the FP64 pipe
Rates are sample-steps/s = C W M lam / time.  The FP64 FMA roof comes from profiles/microbench (as in bench.py); the
kernel's FP64 instructions per sample-step are counted in its SASS (the lam = 1 sample loop, and for lam > 1 the
dynamics step loop plus the per-sample accumulation).
"""
import argparse
import collections
import ctypes
import json
import os
import re
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import random_envs_b200 as renv  # noqa: E402
import sass_stats  # noqa: E402
from random_envs_b200 import _device, build as lib_build  # noqa: E402

XI = (12.0, 1.5, 0.2, 0.7)
EPS = 2e-4
W = 8192
TAU, PML, FORCE = 0.02, 0.05, 10.0
FP64 = ("DFMA", "DMUL", "DADD")


def gpu_info():
    info = dict(gpu=torch.cuda.get_device_name(0))
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        info["power_limit_and_max_sm_clock"] = q[0] if q else "unknown"
    except (OSError, subprocess.SubprocessError) as exc:
        info["power_limit_and_max_sm_clock"] = "unknown (%s)" % exc
    return info


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b) / 1e3


def sass_counts():
    """FP64 instructions of the Euler kernel's lam = 1 sample loop (the smallest loop that reads xi from shared memory)
    and of its dynamics step loop for lam > 1 (the largest loop without shared-memory loads nested in a sample loop)."""
    rows = next(r for n, r in sass_stats.functions(lib_build.LIB_PATH).items() if "transition_loglik_kernelILb1" in n)
    loops = []
    for addr, op, rest in rows:
        m = re.search(r"0x([0-9a-f]+)", rest) if op.startswith("BRA") else None
        if m and int(m.group(1), 16) <= addr:
            body = [o for a, o, _ in rows if int(m.group(1), 16) <= a <= addr]
            loops.append(collections.Counter(o.split(".")[0] for o in body))
    sample = min((h for h in loops if h["LDS"] and h["DFMA"]), key=lambda h: sum(h.values()))
    step = max((h for h in loops if not h["LDS"] and h["DFMA"] and not h["SHFL"]), key=lambda h: h["DFMA"])
    fp = lambda h: sum(h[k] for k in FP64)                                 # noqa: E731
    return dict(lam1_sample_loop_fp64=fp(sample), lam1_sample_loop_instructions=sum(sample.values()),
                step_loop_fp64=fp(step), step_loop_instructions=sum(step.values()),
                accumulate_fp64=18, note="accumulate: 4 differences + 4 sums + 10 FMAs per sample")


def fp64_per_sample_step(counts, lam):
    if lam == 1:
        return counts["lam1_sample_loop_fp64"]
    return counts["step_loop_fp64"] + counts["accumulate_fp64"] / lam


def record(n=512, K=40, seed=5):
    env = renv.RandomCartPoleVecEnv(n, dtype="float64", seed=seed, noisy=True, noise_level=1e-4)
    env.set_task(*XI)
    env.reset()
    obs, act, nxt, done = [], [], [], []
    for _ in range(K):
        o = env.obs.clone()
        a = env.sample_actions().clone()
        o2, _, d, _ = env.step(a)
        obs.append(o); act.append(a); nxt.append(o2.clone()); done.append(d.clone())
    obs, nxt = (torch.stack(v, 1).reshape(-1, 4).cpu().numpy() for v in (obs, nxt))
    act, done = (torch.stack(v, 1).reshape(-1).cpu().numpy() for v in (act, done))
    done = done.astype(bool)
    start = np.zeros(n * K, bool)
    start[::K] = True
    start[1:] |= done[:-1]
    keep = ~done
    return obs[keep], act[keep], nxt[keep], np.flatnonzero(start[keep])


def torch_dynamics(s, xi, a, euler):
    """random_cartpole.py:176-196 on float64 tensors (s: (..., 4), xi broadcastable to (..., 4), a: (...))."""
    x, x_dot, th, th_dot = s.unbind(-1)
    g, mc, mp, l = xi.unbind(-1)
    total = mp + mc
    force = torch.where(a == 1, FORCE, -FORCE)
    c, sn = torch.cos(th), torch.sin(th)
    temp = (force + PML * th_dot * th_dot * sn) / total
    th_acc = (g * sn - c * temp) / (l * (4.0 / 3.0 - mp * c * c / total))
    x_acc = temp - PML * th_acc * c / total
    if euler:
        return torch.stack([x + TAU * x_dot, x_dot + TAU * x_acc, th + TAU * th_dot, th_dot + TAU * th_acc], -1)
    x_dot = x_dot + TAU * x_acc
    th_dot = th_dot + TAU * th_acc
    return torch.stack([x + TAU * x_dot, x_dot, th + TAU * th_dot, th_dot], -1)


def torch_loglik(data, windows, xi, lam, euler, out, chunk=1 << 26):
    """out (C, W): the objective in torch float64, chunked so that one (windows, M) slab has <= chunk elements."""
    C, M, _ = xi.shape
    per = max(1, chunk // (M * 4))
    eye = torch.eye(4, dtype=torch.float64, device=xi.device) * EPS
    for c in range(C):
        for w0 in range(0, windows.numel(), per):
            t = windows[w0:w0 + per].long()
            s = data.obs[t].unsqueeze(1).expand(-1, M, 4)
            for k in range(lam):
                s = torch_dynamics(s, xi[c].unsqueeze(0), data.actions[t + k].unsqueeze(1), euler)
            mu = s.mean(1)
            d = s - mu.unsqueeze(1)
            S = d.transpose(1, 2) @ d / (M - 1) + eye
            L = torch.linalg.cholesky(S)
            r = (data.next_obs[t + lam - 1] - mu).unsqueeze(-1)
            z = torch.linalg.solve_triangular(L, r, upper=False).squeeze(-1)
            out[c, w0:w0 + per] = -0.5 * (z * z).sum(-1) - torch.log(torch.diagonal(L, dim1=1, dim2=2)).sum(-1) \
                - 2.0 * np.log(2 * np.pi)
    return out


def fma_peak_f64():
    sys.path.insert(0, os.path.join(ROOT, "profiles", "microbench"))
    import build as microbench_build                                       # noqa: E402
    mb = ctypes.CDLL(microbench_build.build())
    dev = torch.device("cuda", 0)
    sm = torch.cuda.get_device_properties(dev).multi_processor_count
    blocks, threads, iters = sm * 8, 256, 10000
    buf = torch.empty(blocks * threads, dtype=torch.float64, device=dev)
    launch = lambda: mb.renv_fma_peak_f64(ctypes.c_void_p(buf.data_ptr()), blocks, threads, iters, _device.stream_ptr(dev))  # noqa: E731
    assert launch() == 0
    return max(2.0 * blocks * threads * 8 * iters / timed(launch) / 1e12 for _ in range(3))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--torch-cases", default="16:256:1,16:256:5,64:1024:1")
    args = ap.parse_args()
    torch_cases = {tuple(int(v) for v in c.split(":")) for c in args.torch_cases.split(",") if c}
    counts = sass_counts()
    out = dict(gpu_info(), rounds=args.rounds, windows=W, sass=counts, fma_peak_f64_tflops=fma_peak_f64(), cases=[])
    fp64_instr_per_s = out["fma_peak_f64_tflops"] * 1e12 / 2

    obs, act, nxt, starts = record()
    data = renv.TransitionDataset(obs, act, nxt, episode_starts=starts)
    assert data.num_windows(5) >= W
    data._windows = {lam: torch.as_tensor(data.window_starts(lam)[:W], device="cuda") for lam in (1, 5)}
    out["transitions"] = int(data.num_transitions)

    roll = renv.RandomCartPoleVecEnv(1 << 24, dtype="float64", seed=2)
    roll.set_dr_distribution("uniform", [2.0, 20.0, 0.5, 3.0, 0.05, 0.3, 0.1, 1.0])
    roll.set_dr_training(True)
    roll.reset()
    roll.rollout((0.1, 0.1, 1.0, 0.3), 0.0, 10)
    rollout = lambda: roll.rollout((0.1, 0.1, 1.0, 0.3), 0.0, 500)         # noqa: E731

    mean = np.array(XI)
    cases = [(C, M, lam, True) for C in (16, 64) for M in (256, 1024) for lam in (1, 5)] + [(64, 1024, 1, False)]
    for C, M, lam, euler in cases:
        distrs = [list(np.stack([mean * (0.9 + 0.2 * c / C), 0.02 * mean], 1).reshape(-1)) for c in range(C)]
        xi = data.sample_candidates("truncnorm", distrs, num_samples=M, seed=1)
        integ = "euler" if euler else "semi-implicit"
        arms = dict(kernel=lambda: data.log_likelihood(xi, lam=lam, epsilon=EPS, kinematics_integrator=integ),
                    rollout=rollout)
        rec = dict(C=C, M=M, lam=lam, integrator=integ, sample_steps=C * W * M * lam)
        if (C, M, lam) in torch_cases and euler:
            t_out = torch.empty((C, W), dtype=torch.float64, device="cuda")
            arms["torch"] = lambda: torch_loglik(data, data._windows[lam], xi, lam, euler, t_out)
        for fn in arms.values():
            fn()
        torch.cuda.synchronize()
        if "torch" in arms:
            _, ll = data.log_likelihood(xi, lam=lam, epsilon=EPS, kinematics_integrator=integ, per_window=True)
            rel = ((t_out - ll).abs() / ll.abs().clamp(min=1.0)).max()
            rec["torch_check"] = dict(max_rel_diff=float(rel), within_1e_9=bool(rel <= 1e-9))
        times = {k: [] for k in arms}
        for _ in range(args.rounds):
            for k, fn in arms.items():
                times[k].append(timed(fn))
        rec["seconds"] = times
        for k, ts in times.items():
            work = 500 * (1 << 24) if k == "rollout" else C * W * M * lam
            rec[k] = dict(rate_per_s=work / min(ts), spread=max(ts) / min(ts) - 1)
        rec["kernel_over_rollout"] = rec["kernel"]["rate_per_s"] / rec["rollout"]["rate_per_s"]
        per = fp64_per_sample_step(counts, lam)
        rec["fp64_instr_per_sample_step"] = per
        rec["fp64_pipe_fraction"] = rec["kernel"]["rate_per_s"] * per / fp64_instr_per_s
        if "torch" in rec:
            rec["kernel_over_torch"] = rec["kernel"]["rate_per_s"] / rec["torch"]["rate_per_s"]
        out["cases"].append(rec)
        print(json.dumps(dict((k, v) for k, v in rec.items() if k != "seconds")), flush=True)
        del xi
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            json.dump(out, f, indent=1)


if __name__ == "__main__":
    main()
