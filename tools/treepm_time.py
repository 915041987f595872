"""Times TreePM (Engine.treepm_forces_dev) phase by phase with CUDA events: 2^24 Zel'dovich particles from the
engine's own generator in Hilbert storage order, PM meshes of 256^3 and 512^3, theta = 0.5.  Each phase -- the
fixed-physics tree build, the PM long range, the short-range walk -- is the median of --iters calls after two
warm-up calls.  Also reports the walk counters (b200_tree_walk_stats) of the short-range walk next to those of the
periodic fixed walk (b200_tree_set_periodic) at the same theta, that walk's time, and the card's name and power
limit (read-only nvidia-smi query in the same run).

    python tools/treepm_time.py --out profiles/r3_treepm_time.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "lambda-cdm-raytracing_b200", "python"))

STATS = ["nodes_visited", "cell_interactions", "pair_interactions", "pair_slots", "visit_lanes", "visit_lanes_awake"]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    import torch
    import b200grav
    ap = argparse.ArgumentParser()
    ap.add_argument("--ic-grid", type=int, default=256)          # 256^3 = 2^24 particles
    ap.add_argument("--grids", default="256,512")
    ap.add_argument("--theta", type=float, default=0.5)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "treepm_time needs a GPU"
    torch.cuda.set_device(0)
    eng = b200grav.Engine(0)
    box, theta, cap, depth, eps, factor = 100.0, args.theta, 8, 20, 0.01, 4.5
    n = args.ic_grid ** 3
    posm = torch.empty((n, 4), dtype=torch.float32, device="cuda")
    vel = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    eng.zeldovich_ics_dev(posm, vel, grid=args.ic_grid, box=box, origin_shift=box / 2)
    del vel
    perm = torch.empty(n, dtype=torch.int32, device="cuda")
    eng.spatial_order_dev(posm, n, box, perm)
    posm = posm[perm.long()].contiguous()
    del perm
    out = {"card": card(), "n": n, "box": box, "theta": theta, "leaf_cap": cap, "eps": eps, "r_cut_factor": factor,
           "ics": f"Zel'dovich {args.ic_grid}^3, z = 49, seed 12345, Hilbert storage order", "iters": args.iters,
           "runs": []}
    acc = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(4)]
    for G in [int(g) for g in args.grids.split(",")]:
        rs = 1.25 * box / G
        rows = []
        for it in range(args.iters + 2):                             # two warm-up calls: plans, allocations, graphs
            ev[0].record()
            eng.tree_build_fixed_dev(posm, n, cap, depth, eps)
            ev[1].record()
            eng.pm_forces_dev(posm, acc, 0, n, G, box, rs)
            ev[2].record()
            eng.tree_walk_short_dev(acc, 0, n, theta, box, rs, factor * rs)
            ev[3].record()
            torch.cuda.synchronize()
            if it >= 2:
                rows.append([ev[k].elapsed_time(ev[k + 1]) for k in range(3)])
        med = np.median(np.array(rows), 0)
        assert not torch.isnan(acc).any()
        eng.tree_set_counting(True)
        eng.tree_walk_short_dev(acc, 0, n, theta, box, rs, factor * rs)
        stats = eng.tree_walk_stats()
        eng.tree_set_counting(False)
        run = {"grid": G, "r_split": rs, "r_cut": factor * rs, "build_ms": float(med[0]), "pm_ms": float(med[1]),
               "short_walk_ms": float(med[2]), "total_ms": float(med.sum()),
               "short_walk_stats": {k: int(v) for k, v in zip(STATS, stats)}}
        out["runs"].append(run)
        print(json.dumps(run), flush=True)
    # the periodic fixed walk (minimum image, no cut-off) at the same theta, on the same tree
    eng.tree_build_fixed_dev(posm, n, cap, depth, eps)
    eng.tree_set_periodic(box)
    times = []
    for it in range(args.iters + 2):
        ev[0].record()
        eng.tree_walk_dev(acc, 0, n, theta)
        ev[1].record()
        torch.cuda.synchronize()
        if it >= 2:
            times.append(ev[0].elapsed_time(ev[1]))
    eng.tree_set_counting(True)
    eng.tree_walk_dev(acc, 0, n, theta)
    stats = eng.tree_walk_stats()
    eng.tree_set_counting(False)
    eng.tree_set_periodic(0.0)
    out["periodic_walk"] = {"walk_ms": float(np.median(times)), "stats": {k: int(v) for k, v in zip(STATS, stats)}}
    print(json.dumps(out["periodic_walk"]), flush=True)
    eng.close()
    txt = json.dumps(out, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")
    print(txt)


if __name__ == "__main__":
    main()
