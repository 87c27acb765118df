#!/usr/bin/env python
"""bench.py -- DR env-steps/sec of the RandomCartPole-v0 hot path on N B200s (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--dump-outputs DIR]   # this framework (CUDA kernels)
    python bench.py --impl reference [--gpus N] [--steps K] [--warmup W]       # the reference's CPU path (oracle port)
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...           # N > 1: one rank per GPU

One "step" = one pass of the single-step kernel (RandomCartPoleEnv.step + TimeLimit + auto-reset + uniform DR
resample on reset) over one batch of 2^20 envs -- BASELINE.json configs[1].  Per rank, 4 independent batches
(248 MB > 126 MB L2) are stepped round-robin so every launch streams its working set from HBM.  The K timed steps are
captured in a CUDA graph (a 10 us kernel is otherwise bound by the Python/ctypes launch path); after W eager warm-up
steps, the graph is replayed twice back to back and the second replay -- the K steps -- alone is timed between two CUDA
events: `ms_per_step` is that replay / K.  The eager public-API rate over K steps is reported as `value_eager`.

`--dump-outputs DIR` writes what the last timed step returned (obs, reward, done of the batch it stepped; rank 0) as
DIR/<name>.npy.  Every input is seeded, so two builds run with the same arguments can be compared output for output.

The reference arm (`--impl reference`) runs the REFERENCE's own RandomCartPoleEnv objects (oracle/_ref, see
oracle/make_ref.py; the bit-exact port only if those copies are absent) on all host cores for >= 2 s whatever --steps is.

Rank 0 prints ONE JSON line (see the keys at the bottom of main()).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

BYTES_PER_STEP = {"float32": 62, "float64": 114}    # algorithmic bytes per env-step (SURVEY.md section 8d, DESIGN.md)
FLOPS_PER_STEP_ROLLOUT = 43                          # SURVEY.md section 8d: dynamics 34 + linear policy 9
SEARCH = [2.0, 20.0, 0.5, 3.0, 0.05, 0.3, 0.1, 1.0]  # random_cartpole.py:127-132 = BASELINE cfg 1/2 DR
METRIC = "DR env-steps/sec (RandomCartPole-v0 single-step kernel, uniform DR resample on reset)"
UNIT = "env-steps/s"
SPIN_CYCLES = 400000                                 # torch.cuda._sleep before an event-timed region: ~200 us busy stream


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=100)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--envs", type=int, default=1 << 20, help="envs per batch (= per launch)")
    ap.add_argument("--batches", type=int, default=4, help="independent batches per rank, stepped round-robin")
    ap.add_argument("--dtype", default="float32", choices=["float32", "float64"])
    ap.add_argument("--no-extras", action="store_true", help="skip the size sweep / rollout / sampler extras")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-seconds", type=float, default=10.0)
    ap.add_argument("--ref-seconds", type=float, default=4.0, help="wall time of the reference arm's timed region")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed step as DIR/<name>.npy (float32 / float64, <= 64 MB)")
    args = ap.parse_args()
    if args.impl == "b200" and args.steps < 1:
        ap.error("--steps must be >= 1")
    return args


def workload_config(args, world):
    return {"workload": "RandomCartPole-v0 batched %d envs/launch, uniform DR over the search bounds, resample on "
                        "reset, single-step kernel (BASELINE.json configs[1])" % args.envs,
            "envs_per_launch": args.envs, "batches_per_gpu": args.batches,
            "l2_policy": "inputs larger than L2: %d batches x %.0f MB round-robin per GPU"
                         % (args.batches, args.envs * BYTES_PER_STEP[args.dtype] / 1e6),
            "policy": "random (Bernoulli(1/2) uint8 actions, Philox, pre-generated on device)",
            "max_episode_steps": 500, "integrator": "euler", "parallelism": "envs sharded by index, dp%d" % world,
            "outputs": "state (= obs), reward, done, elapsed: the 62 B/env-step of SURVEY 8d; the optional "
                       "TimeLimit.truncated flags (+1 B) and per-env episode counters are off"}


# --------------------------------------------------------------------------------------------------- reference arm
def run_reference(args):
    """Reference arm: the reference's own CPU implementation of the path, all host cores, same metric and config.

    A "step" of this arm is a BLOCK of gym-0.21 SyncVectorEnv steps over procs x 64 scalar envs: the driver's
    `--steps 20` would otherwise time 7 ms.  Every worker steps its envs for max(2 s, ...) of wall time; the value is
    env-steps / the slowest worker's time."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import cpu_bench
    procs = os.cpu_count() or 1
    envs_per_proc = 64
    seconds = max(2.0, args.ref_seconds)
    res = cpu_bench.run(procs, envs_per_proc, steps=0, warmup=max(20, args.warmup), seconds=seconds)
    k = max(1, args.steps)
    line = {"impl": "reference", "metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * res["seconds"] / k,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(args, max(1, args.gpus)),
            "cpu_baseline": {"value": res["value"], "unit": UNIT, "cores": procs, "kind": res["kind"],
                             "sample": res["sample"], "cpu_model": res["cpu_model"], "seconds": res["seconds"],
                             "step": "one of the %d timed steps = %.0f gym-0.21 SyncVectorEnv.step calls over %d procs x %d "
                                     "reference RandomCartPoleEnv objects" % (k, res["steps"] / k, procs, envs_per_proc)},
            "e2e": {"value": res["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)
    return 0


# --------------------------------------------------------------------------------------------------- helpers
class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md clocks line)."""
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.thread = [], None, None
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.QUERY,
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return self
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self, t0=None, t1=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, smax, power, reasons = [], [], [], set()
        for ts, line in self.rows:
            if t0 is not None and not (t0 - 0.05 <= ts <= t1 + 0.15):
                continue
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); smax.append(float(f[2])); power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples in timed region"], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(smax), "power_w_max": max(power), "reasons": sorted(reasons),
                "samples": len(sm)}


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    except Exception:  # noqa: BLE001
        return 6650.0, "fallback (B200_PROFILING.md)"


def ncu_traffic(dtype):
    """Per-launch DRAM bytes of the step kernel from the committed ncu capture, if there is one."""
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get("cartpole_step_%s_1M" % dtype)
    except Exception:  # noqa: BLE001
        return None


def dump_outputs(directory, arrays, limit_bytes=60 << 20):
    """Write `arrays` (name -> tensor whose first dimension is the env) as DIR/<name>.npy.  If they hold more than
    `limit_bytes` (60 MiB: the files stay below 64 MB), the same fixed, seeded sample of env rows is written from each,
    with its row indices as env_index.npy."""
    import numpy as np
    import torch
    n = next(iter(arrays.values())).shape[0]
    row_bytes = sum(a[0].numel() * a.element_size() for a in arrays.values())
    if n * row_bytes > limit_bytes:
        idx = np.sort(np.random.default_rng(0).choice(n, limit_bytes // (row_bytes + 8), replace=False))
        rows = torch.from_numpy(idx)
        arrays = {name: a.index_select(0, rows.to(a.device)) for name, a in arrays.items()}
        arrays["env_index"] = torch.from_numpy(idx.astype(np.float64))
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + ".npy"), a.cpu().numpy())


# --------------------------------------------------------------------------------------------------- b200 arm
def run_b200(args):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly ONE JSON line: anything libraries print there (e.g. "NCCL version ...") goes to stderr
    sys.stdout.flush()
    json_fd = os.dup(1)
    os.dup2(2, 1)

    cpu_baseline, cpu_c1 = None, None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        # before CUDA is initialised in this process; worker processes are forked inside the child
        out = subprocess.run([sys.executable, "-m", "oracle.cpu_bench", "--seconds", str(args.cpu_seconds)], cwd=ROOT,
                             stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True)
        if out.returncode == 0:
            r = json.loads(out.stdout.strip().splitlines()[-1])
            cpu_baseline = {"value": r["value"], "unit": UNIT, "cores": r["cores"], "kind": r["kind"],
                            "sample": r["sample"], "cpu_model": r["cpu_model"], "seconds": r["seconds"]}
        else:
            cpu_baseline = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "failed: " + out.stderr[-200:]}
        # BASELINE.json configs[0] / BASELINE.md "C1": the reference's own single-env demo loop on one host core
        out = subprocess.run([sys.executable, "-m", "oracle.cpu_bench", "--c1"], cwd=ROOT, stdout=subprocess.PIPE,
                             stderr=subprocess.PIPE, text=True)
        cpu_c1 = json.loads(out.stdout.strip().splitlines()[-1]) if out.returncode == 0 else {"failed": out.stderr[-200:]}

    import torch
    import torch.distributed as dist
    import random_envs_b200 as renv
    from random_envs_b200 import _device, _lib

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    renv.load_library()

    def barrier():
        if world > 1:
            dist.barrier(device_ids=[local_rank])

    def max_over_ranks(ms):
        if world == 1:
            return ms
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def timed(fn):
        """barrier + sync | events around fn() | sync + barrier; returns max-over-ranks milliseconds."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier(); torch.cuda.synchronize()
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize(); barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    n, R, A = args.envs, args.batches, 8
    K = args.steps

    def make_batches(tile_ordering):
        envs, actions = [], []
        for b in range(R):
            env = renv.RandomCartPoleVecEnv(n, dtype=args.dtype, device=dev, seed=0, env_id0=(rank * R + b) * n,
                                            track_truncated=False, track_episodes=False, tile_ordering=tile_ordering)
            env.set_dr_distribution("uniform", SEARCH)
            env.set_dr_training(True)
            env.reset()
            acts = []
            for k in range(A):
                a = torch.empty(n, dtype=torch.uint8, device=dev)
                _lib.call("renv_random_actions_u8", _device.ptr(a), n, env.env_id0, 0, k, _device.stream_ptr(dev))
                acts.append(a)
            envs.append(env); actions.append(acts)
        torch.cuda.synchronize()
        return envs, actions

    def stepper(envs, actions, returned=None):
        """step_i(i) steps batch i % R; `returned[b]` keeps what the last step of batch b returned (views of the env's
        buffers, refreshed in place by every later step, graph replays included)."""
        def step_i(i):
            b = i % R
            out = envs[b].step(actions[b][(i // R) % A])
            if returned is not None:
                returned[b] = out
        return step_i

    # the same K steps as one CUDA graph.  `chain`: one stream, launches in stream order.  `branches`: the R
    # independent env batches on R parallel graph branches, so one batch's tail wave overlaps another's head
    # (a 2^20-env launch is only 1.7 waves of CTAs).
    def capture(step_i, parallel):
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
        return g

    def time_graph(graph):
        """Two back-to-back replays of a K-step graph; the second alone is timed between two CUDA events (max over
        ranks, milliseconds).  The first uploads the graph and keeps the GPU busy with the same K steps while the host
        queues the second, and a spin kernel queued before both covers the host's launch latency: the events bracket
        the K steps, not the host (a 20-step graph is only ~0.23 ms of GPU work) and not the ramp of an idle GPU."""
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier(); torch.cuda.synchronize()
        torch.cuda._sleep(SPIN_CYCLES)
        graph.replay()
        e0.record(); graph.replay(); e1.record()
        torch.cuda.synchronize(); barrier()
        return max_over_ranks(e0.elapsed_time(e1))

    bytes_per = BYTES_PER_STEP[args.dtype]

    # ---- (1) the public API as a user drives it: default env (tile-granular step ordering at this size), ONE stream
    envs_t, actions_t = make_batches("auto")
    step_t = stepper(envs_t, actions_t)
    for i in range(max(args.warmup, 3)):
        step_t(i)
    torch.cuda.synchronize()
    ms_eager = timed(lambda: [step_t(i) for i in range(K)])
    chain = capture(step_t, False)
    ms_chain = time_graph(chain)
    del chain

    # ---- (2) the headline: grid-ordered launches, the R independent batches on R parallel graph branches
    envs, actions = make_batches(False)
    returned = {}
    step_g = stepper(envs, actions, returned)
    for i in range(max(args.warmup, 3)):
        step_g(i)
    torch.cuda.synchronize()
    chain_g = capture(step_g, False)
    ms_chain_g = time_graph(chain_g)
    del chain_g
    graph = capture(step_g, True)

    clocks = ClockSampler(local_rank).start() if rank == 0 else None
    t_wall0 = time.time()
    ms = time_graph(graph)
    # what the last timed step returned, copied before anything steps these envs again
    obs_last, reward_last, done_last, _ = returned[(K - 1) % R]
    outputs = {"obs": obs_last.clone(memory_format=torch.contiguous_format), "reward": reward_last.clone(),
               "done": done_last.to(torch.float32)}
    # keep the GPU under the same load for >= 0.5 s so that nvidia-smi gets samples of the timed workload
    while time.time() - t_wall0 < 0.6:
        graph.replay()
    torch.cuda.synchronize()
    t_wall1 = time.time()
    clock_info = clocks.stop(t_wall0, t_wall1) if clocks else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, outputs)
    del outputs
    value = world * n * K / (ms * 1e-3)
    value_eager = world * n * K / (ms_eager * 1e-3)

    # one launch in isolation (sync on both sides, the 4 batches rotating so that it streams from HBM): the number an
    # ncu launch list shows; the amortised figures above overlap consecutive launches
    def bracket(with_kernel, i):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        torch.cuda._sleep(SPIN_CYCLES)  # ~200 us of busy stream: what follows is queued before the GPU gets to it,
        e0.record()                     # so the events bracket the kernel and not the host's launch latency
        if with_kernel:
            step_g(i)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)
    iso = sorted(bracket(True, i) for i in range(40))
    empty = sorted(bracket(False, i) for i in range(40))           # the two event records alone
    iso_us = 1e3 * max_over_ranks(iso[len(iso) // 2] - empty[len(empty) // 2])

    peak, peak_src = measured_peaks()
    per_launch_ms = ms / K
    achieved = bytes_per * n / (per_launch_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "kernel": "cartpole_step_kernel<%s>" % ("float" if args.dtype == "float32" else "double"),
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
                "bytes_per_env_step": bytes_per, "launch_us": per_launch_ms * 1e3, "isolated_launch_us": iso_us,
                "launch_us_note": "launch_us = graph replay / K with consecutive launches overlapping (amortised); "
                                  "isolated_launch_us = one launch alone on the GPU, nothing before or after it to overlap "
                                  "with (event pair behind a spin kernel minus the same pair with nothing in between; it still "
                                  "contains the launch ramp of a cold stream -- the ncu launch list under profiles/ has the "
                                  "kernel-only duration)",
                "traffic": ncu_traffic(args.dtype)}

    def roof(ms_k):
        gbs = bytes_per * n / (ms_k / K * 1e-3) / 1e9
        return {"launch_us": 1e3 * ms_k / K, "achieved": gbs, "frac": gbs / peak}

    # ---- end to end through the public host-buffer API: pinned H2D actions, D2H obs/reward/done every step.
    # The R env batches are stepped round-robin with one step in flight per batch (step_host_async / _wait), so
    # batch b's device->host transfer overlaps batch b+1's host->device transfer and kernel.
    import numpy as np
    k_e2e = max(2 * R, min(max(K, 100), 200))
    host_actions = [a.cpu().numpy() for a in actions[0][:2]]
    del envs_t, actions_t
    torch.cuda.synchronize()

    def e2e_loop(steps):
        checksum = 0
        for i in range(steps):
            env = envs[i % R]
            if i >= R:
                obs, rew, done, _ = env.step_host_wait()      # results of this batch's previous step are on the host
                checksum += int(done[0])
            env.step_host_async(host_actions[i % 2])
        for b in range(min(R, steps)):
            envs[b].step_host_wait()
        return checksum
    e2e_loop(2 * R)
    barrier(); torch.cuda.synchronize()
    t0 = time.perf_counter(); e2e_loop(k_e2e); torch.cuda.synchronize(); t1 = time.perf_counter()
    ms_e2e = max_over_ranks((t1 - t0) * 1e3)
    h2d_bytes, d2h_bytes = envs[0].host_bytes_per_step()     # counted from the tensors the call copies
    e2e_value = world * n * k_e2e / (ms_e2e * 1e-3)
    e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d_bytes,
           "d2h_bytes_per_step": d2h_bytes, "steps": k_e2e, "ms_per_step": ms_e2e / k_e2e,
           "bound": "pcie (device->host copies of obs + done: %.1f GB/s per GPU, %.1f GB/s over the box; a Gen5 x16 link "
                    "gives ~55 GB/s and the host side of this box ~118 GB/s in total with 8 GPUs copying at once, "
                    "profiles/r1/pcie_aggregate_8gpu.txt)" % (e2e_value / world * d2h_bytes / n / 1e9,
                                                             e2e_value * d2h_bytes / n / 1e9),
           "api": "RandomCartPoleVecEnv.step_host_async(numpy uint8 actions) / step_host_wait() -> numpy obs, reward, "
                  "done; %d env batches round-robin, one step in flight per batch; obs + done cross PCIe (done as bits: packed on "
                  "the device by renv_pack_flags_u8, unpacked into the numpy bool array inside step_host_wait), the reward "
                  "(identically 1.0 under auto-reset, random_cartpole.py:207-212) is a constant host array" % R}

    extras = {}
    if not args.no_extras:
        extras = run_extras(args, torch, dist, renv, _device, _lib, dev, rank, world, timed, peak)
        if cpu_c1 is not None:
            extras["cfg1_cpu_reference_single_env"] = cpu_c1

    if world > 1:
        dist.destroy_process_group()
    if rank != 0:
        return 0
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": args.warmup,
            "ms_per_step": per_launch_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32" if args.dtype == "float32" else "f64", "data": "synthetic",
            "config": workload_config(args, world), "clocks": clock_info, "e2e": e2e, "gpu_launches": K,
            "launch_mode": "one CUDA graph of the K = %d cartpole_step_kernel launches, the %d independent env batches on "
                           "%d parallel graph branches (grid-ordered launches); one replay is timed (%.3f ms) directly "
                           "after an untimed one, ms_per_step = replay / %d" % (K, R, R, ms, K),
            "timing": {"steps_timed": K, "region_ms": ms},
            "value_eager": value_eager, "value_graph_single_chain": world * n * K / (ms_chain * 1e-3),
            "single_stream": {"note": "the default env (tile-granular step ordering, include/renv.h progress) on ONE "
                                      "stream: what a plain step() loop over %d env batches gets" % R,
                              "eager_python_loop": roof(ms_eager), "graph_chain": roof(ms_chain),
                              "graph_chain_grid_ordered": roof(ms_chain_g)},
            "roofline_single_chain": roof(ms_chain),
            "roofline": roofline, "cpu_baseline": cpu_baseline, "extras": extras}
    sys.stdout.flush()
    os.write(json_fd, (json.dumps(line) + "\n").encode())
    return 0


def run_extras(args, torch, dist, renv, _device, _lib, dev, rank, world, timed, peak):
    """Other BASELINE configs, each a few hundred ms: size sweep, fp64, fused rollout, sampler sweep, FMA peaks."""
    import ctypes
    out = {}

    def agg(units, ms):
        return world * units / (ms * 1e-3)

    # single-step kernel at working sets far beyond L2 (SURVEY 0.10): 2^24 and 2^26 envs, plus fp64 at 2^24
    for label, n, dtype, steps in (("step_f32_16M", 1 << 24, "float32", 40), ("step_f32_64M", 1 << 26, "float32", 12),
                                   ("step_f64_16M", 1 << 24, "float64", 20)):
        env = renv.RandomCartPoleVecEnv(n, dtype=dtype, device=dev, seed=1, env_id0=rank * n, track_truncated=False, track_episodes=False)
        env.set_dr_distribution("uniform", SEARCH); env.set_dr_training(True); env.reset()
        a = env.sample_actions().clone()
        for _ in range(3):
            env.step(a)
        ms = timed(lambda: [env.step(a) for _ in range(steps)])
        gbs = BYTES_PER_STEP[dtype] * n * steps / (ms * 1e-3) / 1e9
        out[label] = {"env_steps_per_s": agg(n * steps, ms), "launch_us": 1e3 * ms / steps, "gbs_per_gpu": gbs,
                      "frac_of_hbm_peak": gbs / peak, "envs_per_gpu": n}
        del env, a
        torch.cuda.empty_cache()

    # ONE 2^20-env batch stepped repeatedly (what a single training loop does): its 62 MB working set stays in the
    # 126 MB L2, so this is NOT an HBM number -- reported beside the headline, which rotates 4 batches to defeat L2
    n = 1 << 20
    env = renv.RandomCartPoleVecEnv(n, dtype="float32", device=dev, seed=1, env_id0=rank * n, track_truncated=False, track_episodes=False)
    env.set_dr_distribution("uniform", SEARCH); env.set_dr_training(True); env.reset()
    a = env.sample_actions().clone()
    for _ in range(20):
        env.step(a)
    ms = timed(lambda: [env.step(a) for _ in range(400)])
    out["step_f32_1M_single_batch_l2_resident"] = {"env_steps_per_s": agg(n * 400, ms), "launch_us": 1e3 * ms / 400,
                                                   "algorithmic_gbs_per_gpu": 62 * n * 400 / (ms * 1e-3) / 1e9,
                                                   "note": "L2-resident working set; eager step() loop on one stream"}
    del env, a
    torch.cuda.empty_cache()

    # Lean step (renv_cartpole_step_lean_f32): uint16 TimeLimit counter, no reward store: 35 B read + 19 B written = 54 B
    # per env-step; state / done bit-identical to the 62-byte step (tests/test_gpu_step_modes.py).  4 x 2^20 envs
    # round-robin on one stream (default tile-granular ordering) and 2^24 envs.
    n = 1 << 20
    lean = []
    for b in range(4):
        e = renv.RandomCartPoleVecEnv(n, dtype="float32", device=dev, seed=1, env_id0=(rank * 4 + b) * n,
                                      track_truncated=False, track_episodes=False, lean=True)
        e.set_dr_distribution("uniform", SEARCH); e.set_dr_training(True); e.reset()
        lean.append(e)
    a = lean[0].sample_actions().clone()
    for i in range(40):
        lean[i % 4].step(a)
    ms_eager = timed(lambda: [lean[i % 4].step(a) for i in range(800)])
    # the same 4 x 2^20 envs as ONE single-stream CUDA graph of 400 steps (the eager loop above is partly bound by the
    # Python launch path at 11 us per call)
    g = torch.cuda.CUDAGraph()
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        with torch.cuda.graph(g, stream=side):
            for i in range(400):
                lean[i % 4].step(a)
    torch.cuda.current_stream().wait_stream(side)
    g.replay(); torch.cuda.synchronize()
    ms = min(timed(g.replay) for _ in range(5)) * 2.0        # per 800 steps, as the eager figure
    del g
    gbs = 54 * n * 800 / (ms * 1e-3) / 1e9
    out["step_lean_f32_1M_x4_one_stream"] = {"env_steps_per_s": agg(n * 800, ms), "launch_us": 1e3 * ms / 800, "gbs_per_gpu": gbs,
                                             "frac_of_hbm_peak": gbs / peak, "bytes_per_env_step": 54,
                                             "eager_env_steps_per_s": agg(n * 800, ms_eager),
                                             "traffic": (json.load(open(os.path.join(ROOT, "profiles", "traffic.json")))
                                                         .get("cartpole_step_lean_float32_1M"))}
    del lean, a
    torch.cuda.empty_cache()
    n = 1 << 24
    e = renv.RandomCartPoleVecEnv(n, dtype="float32", device=dev, seed=1, env_id0=rank * n, track_truncated=False,
                                  track_episodes=False, lean=True)
    e.set_dr_distribution("uniform", SEARCH); e.set_dr_training(True); e.reset()
    a = e.sample_actions().clone()
    for _ in range(3):
        e.step(a)
    ms = timed(lambda: [e.step(a) for _ in range(40)])
    gbs = 54 * n * 40 / (ms * 1e-3) / 1e9
    out["step_lean_f32_16M"] = {"env_steps_per_s": agg(n * 40, ms), "launch_us": 1e3 * ms / 40, "gbs_per_gpu": gbs,
                                "frac_of_hbm_peak": gbs / peak, "bytes_per_env_step": 54, "envs_per_gpu": n}
    del e, a
    torch.cuda.empty_cache()

    # BASELINE.json configs[0] through the drop-in gym env (one env, one launch per step): the scalar API's latency
    if rank == 0:
        genv = renv.gym.make("RandomCartPole-v0")
        genv.set_dr_distribution("uniform", SEARCH); genv.set_dr_training(True)
        genv.seed(0); genv.action_space.seed(0)
        genv.reset()
        for _ in range(200):
            _, _, d, _ = genv.step(genv.action_space.sample())
            if d:
                genv.reset()
        t0 = time.perf_counter()
        steps_c1, episodes = 10000, 0
        for _ in range(steps_c1):
            _, _, d, _ = genv.step(genv.action_space.sample())
            if d:
                genv.reset(); episodes += 1
        dt = time.perf_counter() - t0
        out["cfg1_gpu_dropin_single_env"] = {"env_steps_per_s": steps_c1 / dt, "us_per_step": 1e6 * dt / steps_c1,
                                             "episodes": episodes, "mean_episode_length": steps_c1 / max(1, episodes),
                                             "api": "gym.make('RandomCartPole-v0').step(a): the test_random_policy.py loop, "
                                                    "10000 steps incl. resets with uniform DR resample"}
        genv.close()

    # Noisy variant (SURVEY 8f rank 2): +16 B/env-step for the separate obs rows, one Philox block + Box-Muller per env
    n = 1 << 24
    env = renv.RandomCartPoleVecEnv(n, dtype="float32", device=dev, seed=1, env_id0=rank * n, track_truncated=False,
                                    track_episodes=False, noisy=True, noise_level=1e-4)
    env.set_dr_distribution("uniform", SEARCH); env.set_dr_training(True); env.reset()
    a = env.sample_actions().clone()
    for _ in range(3):
        env.step(a)
    ms = timed(lambda: [env.step(a) for _ in range(40)])
    gbs = (BYTES_PER_STEP["float32"] + 16) * n * 40 / (ms * 1e-3) / 1e9
    out["step_f32_noisy_16M"] = {"env_steps_per_s": agg(n * 40, ms), "launch_us": 1e3 * ms / 40, "gbs_per_gpu": gbs,
                                 "frac_of_hbm_peak": gbs / peak, "envs_per_gpu": n, "bytes_per_env_step": 78}
    del env, a
    torch.cuda.empty_cache()

    # FP32 / FP64 FMA peaks for the rollout roofline and the Philox issue roof of the samplers (micro-benchmarks that
    # live outside the product library: profiles/microbench/)
    sm = torch.cuda.get_device_properties(dev).multi_processor_count
    mb = ctypes.CDLL(os.path.join(ROOT, "profiles", "microbench", "librenv_microbench.so"))
    peaks = {}
    for suffix, dt, iters in (("f32", torch.float32, 20000), ("f64", torch.float64, 10000)):
        blocks, threads = sm * 8, 256
        buf = torch.empty(blocks * threads, dtype=dt, device=dev)
        fn = getattr(mb, "renv_fma_peak_" + suffix)
        launch = lambda: fn(ctypes.c_void_p(buf.data_ptr()), blocks, threads, iters, _device.stream_ptr(dev))  # noqa: E731
        assert launch() == 0; torch.cuda.synchronize()
        ms = timed(launch)
        peaks[suffix] = 2.0 * blocks * threads * 8 * iters / (ms * 1e-3) / 1e12
    out["fma_peak_tflops"] = peaks
    blocks, threads, iters = sm * 8, 256, 2000
    buf = torch.empty(blocks * threads * 4, dtype=torch.int32, device=dev)
    launch = lambda: mb.renv_philox_peak(ctypes.c_void_p(buf.data_ptr()), blocks, threads, iters, ctypes.c_uint64(1), _device.stream_ptr(dev))  # noqa: E731
    assert launch() == 0; torch.cuda.synchronize()
    ms = timed(launch)
    philox_blocks_per_s = blocks * threads * iters / (ms * 1e-3)
    out["philox_peak"] = {"blocks_per_s": philox_blocks_per_s, "fp32_output_gbs": philox_blocks_per_s * 16 / 1e9,
                          "note": "Philox4x32-10 with nothing else in the loop: the int-multiply issue roof of the samplers"}

    # BASELINE configs[3]: fused 500-step rollout, 2^24 envs per GPU, linear policy, + the stats all-gather
    # (w = None: the random policy of BASELINE configs[0] / test_random_policy.py, one Philox block per env-step)
    for label, dtype, w in (("rollout_f32_survive", "float32", (0.1, 0.1, 1.0, 0.3)), ("rollout_f32_resetheavy", "float32", (0.0, 0.0, 1.0, 0.0)),
                            ("rollout_f64_survive", "float64", (0.1, 0.1, 1.0, 0.3)), ("rollout_f32_random_policy", "float32", None)):
        n, K = 1 << 24, 500
        env = renv.RandomCartPoleVecEnv(n, dtype=dtype, device=dev, seed=2, env_id0=rank * n)
        env.set_dr_distribution("uniform", SEARCH); env.set_dr_training(True); env.reset()
        env.rollout(w, 0.0, 10)
        renv.allgather_stats(env.stats_tensor)      # untimed: the first collective sets up NCCL's communicator / channels
        env.reset_stats()

        def it():
            env.rollout(w, 0.0, K)
            combined, _ = renv.allgather_stats(env.stats_tensor)      # the one collective: 6 doubles per rank
            return combined
        ms = timed(it)
        st = renv.summarize_stats(renv.allgather_stats(env.stats_tensor)[0].cpu().numpy())
        rate = agg(n * K, ms)
        pk = peaks["f32" if dtype == "float32" else "f64"]
        out[label] = {"env_steps_per_s": rate, "ms": ms, "envs_per_gpu": n, "K": K, "policy_w": list(w) if w else "random",
                      "algorithmic_tflops_per_gpu": rate / world * FLOPS_PER_STEP_ROLLOUT / 1e12,
                      "frac_of_fma_peak": rate / world * FLOPS_PER_STEP_ROLLOUT / 1e12 / pk,
                      "episodes": st["episodes"], "mean_return": st["mean_return"]}
        del env
        torch.cuda.empty_cache()

    # BASELINE configs[2]: truncnormal DR, 2^26 envs IN TOTAL sharded by index over the ranks (strong scaling), one
    # 500-step iteration of the fused rollout + the all-gather of the return statistics (SURVEY 8d cfg 3)
    total, K = 1 << 26, 500
    lo_id, hi_id = renv.shard_range(total, rank, world)
    env = renv.RandomCartPoleVecEnv(hi_id - lo_id, dtype="float32", device=dev, seed=3, env_id0=lo_id)
    env.set_dr_distribution("truncnorm", [9.8, 0.98, 1.0, 0.1, 0.2, 0.02, 0.5, 0.05]); env.set_dr_training(True); env.reset()
    w = (0.1, 0.1, 1.0, 0.3)
    env.rollout(w, 0.0, 10)
    renv.allgather_stats(env.stats_tensor)
    env.reset_stats()
    ms = timed(lambda: (env.rollout(w, 0.0, K), renv.allgather_stats(env.stats_tensor)))
    st = renv.summarize_stats(renv.allgather_stats(env.stats_tensor)[0].cpu().numpy())
    out["cfg3_truncnorm_64M_sharded_rollout"] = {"env_steps_per_s": total * K / (ms * 1e-3), "ms": ms, "envs_total": total,
                                                 "envs_per_gpu": hi_id - lo_id, "K": K, "scaling": "strong",
                                                 "episodes": st["episodes"], "mean_return": st["mean_return"]}
    del env
    torch.cuda.empty_cache()

    # BASELINE configs[4]: humanoid 30-dim sampler sweep, 2^24 samples per call
    nu = list(renv.HUMANOID_NOMINAL)
    n = 1 << 24
    for dr_type in ("uniform", "gaussian", "truncnorm", "fullgaussian"):
        s = renv.TaskSampler("RandomHumanoid-v0")
        distr = []
        for v in nu:
            distr += [0.5 * v, 1.5 * v] if dr_type == "uniform" else [v, 0.1 * v]
        if dr_type == "fullgaussian":      # SURVEY 8f rank 1: correlated normal in the normalised [0, 4] space (dim x dim mat-vec)
            import numpy as np
            a = np.random.RandomState(0).randn(30, 30) * 0.1
            distr = {"mean": np.full(30, 2.0), "cov": a @ a.T + 0.05 * np.eye(30)}
        s.set_dr_distribution(dr_type, distr)
        buf = torch.empty((n, 30), dtype=torch.float32, device=dev)
        s.sample_tasks_tensor(n, out=buf); torch.cuda.synchronize()
        ms = timed(lambda: [s.sample_tasks_tensor(n, out=buf) for _ in range(3)]) / 3
        gbs = n * 30 * 4 / (ms * 1e-3) / 1e9
        # every 30-dim sample costs 8 Philox blocks (7.5 rounded up), i.e. 128 B of raw draws for 120 B written
        philox_gbs = out["philox_peak"]["fp32_output_gbs"] * 30.0 / 32.0
        out["sampler_f32_humanoid30_" + dr_type] = {"xi_per_s": agg(n, ms), "ms": ms, "gbs_per_gpu": gbs,
                                                    "frac_of_hbm_peak": gbs / peak,
                                                    "bound": "tensor + philox" if dr_type == "fullgaussian" else "philox int-mul issue",
                                                    "frac_of_philox_roof": gbs / philox_gbs}
        del buf
    torch.cuda.empty_cache()
    return out


def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
