"""Times the periodic particle-mesh force (b200_pm_forces_dev) phase by phase with CUDA events: 2^24 Zel'dovich
particles from the engine's own generator, meshes of 128^3 / 256^3 / 512^3, the particles stored in random and in
Hilbert order.  Reports the bytes each phase has to move against the measured HBM bandwidth, CIC contributions
deposited per second, the card's name and power limit (read-only nvidia-smi query in the same run), and compares a
sample of 4096 targets against the float64 numpy restatement (oracle/pm_np.py).

    python tools/pm_time.py --out profiles/r3_pm_time.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "lambda-cdm-raytracing_b200", "python"))

PHASES = ["deposit", "convert", "r2c", "kspace", "c2r_x3", "interp"]


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def phase_bytes(n, G):
    """Least HBM traffic of each phase (each array read or written once)."""
    cells = G ** 3
    modes = G * G * (G // 2 + 1)
    return {
        "deposit": 8 * cells + 2 * 16 * n + 8 * cells,    # clear + mass bound and deposit reads + mesh written once
        "convert": 8 * cells + 4 * cells,
        "r2c": 4 * cells + 8 * modes,
        "kspace": 8 * modes + 3 * 8 * modes,
        "c2r_x3": 3 * (8 * modes + 4 * cells),
        "interp": 16 * n + 12 * n + 3 * 4 * cells,
    }


def main():
    import torch
    import b200grav
    import bench
    from oracle import pm_np
    ap = argparse.ArgumentParser()
    ap.add_argument("--ic-grid", type=int, default=256)          # 256^3 = 2^24 particles
    ap.add_argument("--grids", default="128,256,512")
    ap.add_argument("--iters", type=int, default=10)
    ap.add_argument("--check-grids", default="128,256", help="meshes compared against numpy (float64 host memory)")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "pm_time needs a GPU"
    torch.cuda.set_device(0)
    eng = b200grav.Engine(0)
    box = 100.0
    n = args.ic_grid ** 3
    posm = torch.empty((n, 4), dtype=torch.float32, device="cuda")
    vel = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    eng.zeldovich_ics_dev(posm, vel, grid=args.ic_grid, box=box, origin_shift=box / 2)
    perm = torch.empty(n, dtype=torch.int32, device="cuda")
    eng.spatial_order_dev(posm, n, box, perm)
    orders = {"random": posm[torch.randperm(n, device="cuda")].contiguous(), "hilbert": posm[perm.long()].contiguous()}
    del vel
    peak, peak_src = bench.hbm_peak()
    out = {"card": card(), "n": n, "box": box, "ics": f"Zel'dovich {args.ic_grid}^3, z = 49, seed 12345",
           "hbm_peak_gbs": peak, "hbm_peak_source": peak_src, "iters": args.iters, "runs": []}
    acc = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    for G in [int(g) for g in args.grids.split(",")]:
        rs = 1.25 * box / G
        for name, pm in orders.items():
            for _ in range(2):                                     # warm-up: plans, allocations, module load
                eng.pm_forces_dev(pm, acc, grid=G, box=box, r_split=rs)
            torch.cuda.synchronize()
            eng.set_timing(True)
            rows = []
            for _ in range(args.iters):
                eng.pm_forces_dev(pm, acc, grid=G, box=box, r_split=rs)
                rows.append(eng.pm_phase_ms())
            eng.set_timing(False)
            med = np.median(np.array(rows), 0)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(args.iters):
                eng.pm_forces_dev(pm, acc, grid=G, box=box, r_split=rs)
            e1.record()
            torch.cuda.synchronize()
            call_ms = e0.elapsed_time(e1) / args.iters
            by = phase_bytes(n, G)
            run = {"grid": G, "order": name, "r_split": rs, "call_ms_untimed": call_ms,
                   "call_ms_phase_events": float(med[6]), "phases": {}}
            for k, ph in enumerate(PHASES):
                ms = float(med[k])
                run["phases"][ph] = {"ms": ms, "min_bytes": by[ph], "gbs": by[ph] / (ms * 1e-3) / 1e9,
                                     "hbm_frac": by[ph] / (ms * 1e-3) / 1e9 / peak}
            run["cic_contributions_per_s"] = 8 * n / (float(med[0]) * 1e-3)
            out["runs"].append(run)
            print(json.dumps(run), flush=True)
    # accuracy at the timed size: every storage order gives the same bits, so one order is compared
    pos = orders["hilbert"][:, :3].double().cpu().numpy()
    mass = orders["hilbert"][:, 3].double().cpu().numpy()
    pick = np.random.default_rng(0).choice(n, 4096, replace=False)
    out["check"] = []
    for G in [int(g) for g in args.check_grids.split(",") if g]:
        rs = 1.25 * box / G
        eng.pm_forces_dev(orders["hilbert"], acc, grid=G, box=box, r_split=rs)
        a_dev = acc[torch.from_numpy(pick).cuda()].double().cpu().numpy()
        a_np = pm_np.pm_forces(pos, mass, pos[pick], G, box, rs)
        err = float(np.linalg.norm(a_dev - a_np) / np.linalg.norm(a_np))
        out["check"].append({"grid": G, "targets": 4096, "rel_l2_vs_pm_np": err})
        print(json.dumps(out["check"][-1]), flush=True)
    eng.close()
    txt = json.dumps(out, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(txt + "\n")
    print(txt)


if __name__ == "__main__":
    main()
