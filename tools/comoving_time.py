"""Times one comoving TreePM step of ComovingSimulation (DESIGN 3.13) phase by phase with CUDA events: 2^24
Zel'dovich particles (256^3, z = 49) from the engine's own generator, PM mesh 256^3, r_s = 1.25 h, theta = 0.5,
r_cut = 4.5 r_s.  A step is: fused half-kick + drift (leapfrog), tree build, PM, short-range walk, closing
half-kick; each phase is the median over --iters steps after two warm-up steps, and so is the whole step (host
clock around the step, ending in a synchronise).  Also the cost of one b200_treepm_energy_dev call, and the card's
name and power limit (read-only nvidia-smi query in the same run).

    python tools/comoving_time.py --out profiles/r3_comoving_time.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "lambda-cdm-raytracing_b200", "python"))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def main():
    import torch
    import b200grav
    ap = argparse.ArgumentParser()
    ap.add_argument("--ic-grid", type=int, default=256)          # 256^3 = 2^24 particles
    ap.add_argument("--pm-grid", type=int, default=256)
    ap.add_argument("--theta", type=float, default=0.5)
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "comoving_time needs a GPU"
    torch.cuda.set_device(0)
    eng = b200grav.Engine(0)
    box, eps = 100.0, 0.01
    pos, mom, mass, a0 = b200grav.comoving_zeldovich_dev(eng, grid=args.ic_grid, box=box, z_initial=49.0)
    sim = b200grav.ComovingSimulation(eng, pos, mom, mass, box, a0, force="treepm", pm_grid=args.pm_grid,
                                      theta=args.theta, eps=eps)
    del pos, mom, mass
    n, G, rs = sim.n, sim.pm_grid, sim.r_split
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(6)]
    scale = np.geomspace(a0, 0.05, 2 * (args.iters + 2) + 1)
    sim.compute_forces()
    rows = []
    for it in range(args.iters + 2):                                # phases of one step, as ComovingSimulation.step
        a1 = scale[it + 1]
        am = np.sqrt(sim.a * a1)
        drift, _ = eng.comoving_kdk_factors(sim.a, a1, *sim.cosmo)
        k0, k1 = eng.comoving_kdk_factors(sim.a, am, *sim.cosmo)[1], eng.comoving_kdk_factors(am, a1, *sim.cosmo)[1]
        ev[0].record()
        eng.leapfrog_dev(sim.posm, sim.mom, sim.acc, n, 1, np.float32(k0), 1.0, np.float32(drift), box)
        ev[1].record()
        eng.tree_build_fixed_dev(sim.posm, n, sim.leaf_cap, sim.max_depth, eps)
        ev[2].record()
        eng.pm_forces_dev(sim.posm, sim.acc, 0, n, G, box, rs)
        ev[3].record()
        eng.tree_walk_short_dev(sim.acc, 0, n, sim.theta, box, rs, 4.5 * rs)
        ev[4].record()
        eng.leapfrog_dev(sim.posm, sim.mom, sim.acc, n, 1, np.float32(k1), 1.0, 0.0, box)
        ev[5].record()
        torch.cuda.synchronize()
        sim.a = a1
        if it >= 2:
            rows.append([ev[k].elapsed_time(ev[k + 1]) for k in range(5)])
    med = np.median(np.array(rows), 0)
    steps = []
    for it in range(args.iters + 2):                                # whole steps through the public class
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        sim.step(scale[args.iters + 3 + it])
        torch.cuda.synchronize()
        if it >= 2:
            steps.append(1e3 * (time.perf_counter() - t0))
    energy = []
    for it in range(args.iters + 2):                                # the tree of the current positions is built
        t0 = time.perf_counter()
        sim.energies()
        if it >= 2:
            energy.append(1e3 * (time.perf_counter() - t0))
    assert torch.isfinite(sim.posm).all() and not eng.tree_overflowed()
    out = {"card": card(), "n": n, "box": box, "pm_grid": G, "r_split": rs, "r_cut": 4.5 * rs, "theta": sim.theta,
           "eps": eps, "leaf_cap": sim.leaf_cap, "ics": f"Zel'dovich {args.ic_grid}^3, z = 49, seed 12345",
           "iters": args.iters, "a_range": [float(a0), float(sim.a)],
           "phase_ms": {"kick_drift": float(med[0]), "tree_build": float(med[1]), "pm": float(med[2]),
                        "short_walk": float(med[3]), "kick": float(med[4]), "sum": float(med.sum())},
           "step_ms": float(np.median(steps)), "treepm_energy_ms": float(np.median(energy))}
    eng.close()
    txt = json.dumps(out, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")
    print(txt)


if __name__ == "__main__":
    main()
