"""Time the periodic direct sum at the production configuration (2^20 particles in [0, 100), eps = 0.01: the
fixed-point x/y path) for one or more builds of libb200grav.so, alternating them call by call so that they share the
card's clock and load.  Prints one JSON line: the card, its power limit, and per library the median and spread of
the CUDA-event time of a whole b200_direct_forces_dev call.

  python tools/direct_periodic_time.py [--reps 20] LIB [LIB ...]
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "lambda-cdm-raytracing_b200", "python"))
import b200grav  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("libs", nargs="+")
    ap.add_argument("--n", type=int, default=1 << 20)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    rng = np.random.default_rng(42)
    pos = rng.uniform(0.0, 100.0, (args.n, 3)).astype(np.float32)
    posm = torch.from_numpy(np.concatenate([pos, np.ones((args.n, 1), np.float32)], 1)).cuda()
    engines = [b200grav.Engine(0, lib=b200grav.load_library(os.path.abspath(p))) for p in args.libs]
    outs = [torch.empty((args.n, 3), dtype=torch.float32, device="cuda") for _ in engines]
    times = [[] for _ in engines]
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for rep in range(args.reps + 2):
        for k, e in enumerate(engines):
            ev0.record()
            e.direct_forces_dev(posm, outs[k], 0, args.n, eps=0.01, box=100.0)
            ev1.record()
            ev1.synchronize()
            if rep >= 2:                                    # two warm-up rounds per library
                times[k].append(ev0.elapsed_time(ev1))
    same = all(torch.equal(outs[0], o) for o in outs[1:])
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip()
    res = {"card": smi, "n": args.n, "eps": 0.01, "box": 100.0, "outputs_bitwise_equal": same,
           "ms": {os.path.basename(p): {"median": float(np.median(t)), "min": float(np.min(t)),
                                        "max": float(np.max(t))} for p, t in zip(args.libs, times)}}
    print(json.dumps(res))
    for e in engines:
        e.close()


if __name__ == "__main__":
    main()
