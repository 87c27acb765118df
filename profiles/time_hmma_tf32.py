"""Throughput and latency of mma.sync TF32 (HMMA.1688.F32.TF32) on this GPU: compiles profiles/exp/hmma_tf32.cu into a
temporary directory, runs it and writes its JSON lines (plus the GPU name and power limit) to --out.

    python profiles/time_hmma_tf32.py [--out FILE]

DESIGN.md section 4.9 compares the MLP rollout's HMMA rate with these numbers.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "profiles"))

from time_mlp_rollout import gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    nvcc = os.environ.get("NVCC", "/usr/local/cuda/bin/nvcc")
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "hmma_tf32")
        subprocess.run([nvcc, "-O3", "-std=c++17", "-gencode", "arch=compute_100a,code=sm_100a", "-o", exe,
                        os.path.join(ROOT, "profiles", "exp", "hmma_tf32.cu")], check=True)
        lines = subprocess.run([exe], check=True, capture_output=True, text=True).stdout.splitlines()
    rows = [json.loads(line) for line in lines]
    for r in rows:
        print(json.dumps(r))
    if args.out:
        with open(args.out, "w") as f:
            json.dump(dict(gpu_info(), rows=rows), f, indent=1)


if __name__ == "__main__":
    main()
