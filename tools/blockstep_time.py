"""Times one PM step with block time steps (ComovingSimulation(max_bins=4), DESIGN 3.14) against eight global steps
of its finest sub-step, on 2^24 Zel'dovich particles (256^3, z = 49, the engine's generator) evolved with global
TreePM steps to a clustered state.  PM mesh 256^3, r_s = 1.25 h, theta = 0.5, r_cut = 4.5 r_s, eps = 0.01.

The block step is run twice from the same state: once phase by phase from Engine calls in the order of
ComovingSimulation.step, with CUDA events around every pass, drift, tree build, PM and active walk (the result is
checked bit-equal to the second run), and once through ComovingSimulation.step under a host clock ending in a
synchronise; the eight global steps likewise through the class.  Records bin occupancy, short-range target
evaluations, and the card's name and power limit (read-only nvidia-smi query in the same run).

    python tools/blockstep_time.py --out profiles/r3_blockstep_time.json
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
    ap.add_argument("--ic-grid", type=int, default=256)
    ap.add_argument("--pm-grid", type=int, default=256)
    ap.add_argument("--a-clustered", type=float, default=0.5)
    ap.add_argument("--evolve-steps", type=int, default=40)
    ap.add_argument("--dlna", type=float, default=0.02)
    ap.add_argument("--max-bins", type=int, default=4)
    ap.add_argument("--eta", type=float, default=0.025)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "blockstep_time needs a GPU"
    torch.cuda.set_device(0)
    eng = b200grav.Engine(0)
    box, eps, theta, cosmo = 100.0, 0.01, 0.5, (0.31, 0.0, 0.69)
    pos, mom, mass, a0 = b200grav.comoving_zeldovich_dev(eng, grid=args.ic_grid, box=box, z_initial=49.0)
    mk = lambda p, q, a, mb: b200grav.ComovingSimulation(eng, p, q, mass, box, a, force="treepm",
                                                         pm_grid=args.pm_grid, theta=theta, eps=eps, cosmo=cosmo,
                                                         max_bins=mb, eta=args.eta)
    sim = mk(pos, mom, a0, 1)
    del pos, mom
    t0 = time.perf_counter()
    for a in np.geomspace(a0, args.a_clustered, args.evolve_steps + 1)[1:]:
        sim.step(a)
    torch.cuda.synchronize()
    evolve_s = time.perf_counter() - t0
    pos0, mom0 = sim.posm[:, :3].clone(), sim.mom.clone()
    del sim
    a_s = args.a_clustered
    a_e = a_s * np.exp(args.dlna)
    n, G = pos0.shape[0], args.pm_grid

    # phase by phase, as ComovingSimulation.step
    t = mk(pos0, mom0, a_s, args.max_bins)
    t.compute_forces()
    ph = {"pass": 0.0, "drift": 0.0, "tree_build": 0.0, "pm": 0.0, "active_walk": 0.0}
    counts = {"passes": 0, "builds": 0, "walks": 0}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]

    def timed(name, fn):
        ev[0].record()
        r = fn()
        ev[1].record()
        torch.cuda.synchronize()
        ph[name] += ev[0].elapsed_time(ev[1])
        return r
    Lb = args.max_bins - 1
    S = 1 << Lb
    kicks, nodes = b200grav.block_factor_table(eng.L, a_s, a_e, args.max_bins, cosmo)
    factors = torch.from_numpy(kicks.astype(np.float32)).cuda()
    dlna = float(np.log(a_e / a_s))
    occupancy = []
    timed("pass", lambda: t._pass(0, nodes[0], factors, dlna))
    counts["passes"] += 1
    occupancy.append([0] + t.bin_counts[:args.max_bins].tolist())
    k = 0
    rs = t.r_split
    while k < S:
        k1 = b200grav.next_sync_point(k, t.bin_counts, args.max_bins)
        drift, _ = eng.comoving_kdk_factors(nodes[k], nodes[k1], *cosmo)
        timed("drift", lambda: eng.leapfrog_dev(t.posm, t.mom, t.acc, n, 0, 0.0, 1.0, np.float32(drift), box))
        k = k1
        timed("tree_build", lambda: eng.tree_build_fixed_dev(t.posm, n, t.leaf_cap, t.max_depth, eps))
        counts["builds"] += 1
        if k == S:
            timed("pm", lambda: eng.pm_forces_dev(t.posm, t.acc_long, 0, n, G, box, rs))
        t.short_targets += timed("active_walk", lambda: eng.tree_walk_short_active_dev(
            t.bins, n, k, args.max_bins, theta, box, rs, 4.5 * rs, t.acc_short))
        counts["walks"] += 1
        timed("pass", lambda: t._pass(k, nodes[k], factors, dlna))
        counts["passes"] += 1
        occupancy.append([k] + t.bin_counts[:args.max_bins].tolist())
    phased_targets = t.short_targets - n

    # whole steps through the class
    def whole(mb, n_steps):
        s = mk(pos0, mom0, a_s, mb)
        s.compute_forces()
        s.short_targets = 0
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for a in np.geomspace(a_s, a_e, n_steps + 1)[1:]:
            s.step(a)
        torch.cuda.synchronize()
        return s, 1e3 * (time.perf_counter() - t0)
    blk, blk_ms = whole(args.max_bins, 1)
    assert torch.equal(blk.posm, t.posm) and torch.equal(blk.mom, t.mom), "phase-timed step differs from step()"
    blk_targets, blk_bins = blk.short_targets, blk.bin_counts[:args.max_bins].tolist()
    del blk, t
    glb, glb_ms = whole(1, S)
    glb_targets = glb.short_targets
    assert torch.isfinite(glb.posm).all() and not eng.tree_overflowed()
    del glb
    out = {"card": card(), "n": n, "box": box, "pm_grid": G, "r_split": rs, "r_cut": 4.5 * rs, "theta": theta,
           "eps": eps, "ics": f"Zel'dovich {args.ic_grid}^3, z = 49, seed 12345, {args.evolve_steps} global TreePM "
                              f"steps to a = {a_s}", "evolve_s": evolve_s,
           "pm_step": {"a": [a_s, float(a_e)], "dlna": args.dlna, "max_bins": args.max_bins, "eta": args.eta},
           "block": {"step_ms": blk_ms, "phase_ms": {k_: round(v, 3) for k_, v in ph.items()},
                     "phase_sum_ms": sum(ph.values()), "launch_counts": counts,
                     "occupancy_after_each_sync_point": occupancy, "final_bins": blk_bins,
                     "short_targets": blk_targets, "short_targets_phased": phased_targets},
           f"global_{S}_steps": {"step_ms_total": glb_ms, "short_targets": glb_targets}}
    eng.close()
    txt = json.dumps(out, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")
    print(txt)


if __name__ == "__main__":
    main()
