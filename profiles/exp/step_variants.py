"""A/B timing of the fp32 auto-reset step kernel: grid- vs tile-granular step ordering; 62 B vs lean 54 B.

    python profiles/exp/step_variants.py [--tag name]

Prints one JSON object per (kernel, mode).  Modes: `chain` = one CUDA graph of K launches on ONE stream over 4 rotating
2^20-env batches (what a plain step() loop does, minus the Python launch path); `branches` = the same with the 4
batches on 4 parallel graph branches (bench.py's headline); `eager` = the Python step() loop; `lone` = one 2^20-env
batch stepped repeatedly (L2-resident); `big` = 2^24 envs.
"""
import argparse
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__)))))

ap = argparse.ArgumentParser()
ap.add_argument("--tag", default="default")
ap.add_argument("--K", type=int, default=400)
ap.add_argument("--reps", type=int, default=5)
ap.add_argument("--batches", type=int, default=4)
ap.add_argument("--modes", default="chain,branches,eager,lone,big")
ap.add_argument("--kernels", default="grid,tile,grid_lean,tile_lean")
args = ap.parse_args()

import torch  # noqa: E402

import random_envs_b200 as renv  # noqa: E402
from random_envs_b200 import _device, _lib  # noqa: E402

SEARCH = [2.0, 20.0, 0.5, 3.0, 0.05, 0.3, 0.1, 1.0]
dev = torch.device("cuda", 0)
torch.cuda.set_device(dev)
PEAK = 6552.0
try:
    PEAK = float(json.load(open(os.path.join(os.path.dirname(__file__), "..", "..", "MEASURED_PEAKS.json")))["hbm_gbs"])
except Exception:  # noqa: BLE001
    pass


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record(); fn(); e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def make(n, R, lean, tile):
    envs, acts = [], []
    for b in range(R):
        env = renv.RandomCartPoleVecEnv(n, dtype="float32", device=dev, seed=0, env_id0=b * n, track_truncated=False,
                                        track_episodes=False, lean=lean, tile_ordering=tile)
        env.set_dr_distribution("uniform", SEARCH); env.set_dr_training(True); env.reset()
        aa = []
        for k in range(8):
            a = torch.empty(n, dtype=torch.uint8, device=dev)
            _lib.call("renv_random_actions_u8", _device.ptr(a), n, env.env_id0, 0, k, _device.stream_ptr(dev))
            aa.append(a)
        envs.append(env); acts.append(aa)
    torch.cuda.synchronize()
    return envs, acts


def capture(step_i, K, R, parallel):
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            if not parallel:
                for i in range(K):
                    step_i(i)
            else:
                lanes = [torch.cuda.Stream(device=dev) for _ in range(R)]
                for b, lane in enumerate(lanes):
                    lane.wait_stream(side)
                    with torch.cuda.stream(lane):
                        for i in range(b, K, R):
                            step_i(i)
                for lane in lanes:
                    side.wait_stream(lane)
    torch.cuda.current_stream().wait_stream(side)
    g.replay(); torch.cuda.synchronize()
    return g


def report(kernel, mode, n, steps, ms_list, bytes_per):
    ms_list = sorted(ms_list)
    ms = ms_list[len(ms_list) // 2]
    us = 1e3 * ms / steps
    gbs = bytes_per * n / us / 1e3
    print(json.dumps({"tag": args.tag, "kernel": kernel, "mode": mode, "n": n, "us_per_launch": round(us, 3),
                      "us_min": round(1e3 * ms_list[0] / steps, 3), "us_max": round(1e3 * ms_list[-1] / steps, 3),
                      "env_steps_per_s": n / us * 1e6, "gbs": round(gbs, 1), "frac": round(gbs / PEAK, 4),
                      "bytes_per_env_step": bytes_per, "batches": args.batches}), flush=True)


modes = args.modes.split(",")
for kernel in args.kernels.split(","):
    tile, lean = kernel.startswith("tile"), kernel.endswith("lean")
    bytes_per = 54 if lean else 62
    n, R, K = 1 << 20, args.batches, args.K
    envs, acts = make(n, R, lean, tile)

    def step_i(i):
        b = i % R
        envs[b].step(acts[b][(i // R) % 8])
    for i in range(100):
        step_i(i)
    torch.cuda.synchronize()
    if "chain" in modes:
        g = capture(step_i, K, R, False)
        report(kernel, "chain", n, K, [timed(g.replay) for _ in range(args.reps)], bytes_per)
        del g
    if "branches" in modes:
        g = capture(step_i, K, R, True)
        report(kernel, "branches", n, K, [timed(g.replay) for _ in range(args.reps)], bytes_per)
        del g
    if "eager" in modes:
        report(kernel, "eager", n, K, [timed(lambda: [step_i(i) for i in range(K)]) for _ in range(3)], bytes_per)
    if "lone" in modes:
        g = capture(lambda i: envs[0].step(acts[0][i % 8]), K, 1, False)
        report(kernel, "lone_graph", n, K, [timed(g.replay) for _ in range(args.reps)], bytes_per)
        del g
    del envs, acts
    torch.cuda.empty_cache()
    if "big" in modes:
        n = 1 << 24
        envs, acts = make(n, 1, lean, tile)
        for _ in range(5):
            envs[0].step(acts[0][0])
        report(kernel, "big_eager", n, 40, [timed(lambda: [envs[0].step(acts[0][i % 8]) for i in range(40)]) for _ in range(3)],
               bytes_per)
        del envs, acts
        torch.cuda.empty_cache()
