"""Times the Barnes-Hut build and the walk with CUDA events and prints the walk's interaction counters."""
import argparse
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "lambda-cdm-raytracing_b200", "python"))


def main():
    import torch
    import b200grav
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 20)
    ap.add_argument("--dist", default="uniform", choices=["uniform", "box", "clustered"])
    args = ap.parse_args()
    n = args.n
    rng = np.random.default_rng(42)
    if args.dist == "uniform":
        pos = rng.uniform(-50, 50, (n, 3))
    elif args.dist == "box":
        pos = rng.uniform(0, 100, (n, 3))
    else:
        c = rng.uniform(-40, 40, (64, 3))
        pos = np.clip(c[rng.integers(0, 64, n)] + rng.normal(0, 2.0, (n, 3)), -49.9, 49.9)
    posm = torch.from_numpy(np.concatenate([pos, np.ones((n, 1))], 1).astype(np.float32)).cuda()
    eng = b200grav.Engine(0)
    acc = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(3):
        eng.tree_build_dev(posm, n, 100.0, 8, 20)
    torch.cuda.synchronize()
    ev0.record()
    for _ in range(5):
        eng.tree_build_dev(posm, n, 100.0, 8, 20)
    ev1.record()
    torch.cuda.synchronize()
    print(f"n={n} dist={args.dist}  build {ev0.elapsed_time(ev1) / 5:.3f} ms  stats {eng.tree_stats()}")
    eng.set_timing(True)
    best = 1e30
    for _ in range(4):
        eng.tree_walk_dev(acc, 0, n, 0.5)
        torch.cuda.synchronize()
        best = min(best, eng.last_kernel_ms())
    eng.tree_set_counting(True)
    eng.tree_walk_dev(acc, 0, n, 0.5)
    torch.cuda.synchronize()
    cnt = eng.tree_counters()
    st = [int(x) for x in eng.tree_walk_stats()]
    eng.tree_set_counting(False)
    inter = float(cnt[1] + cnt[2])
    print(f"walk {best:8.3f} ms  {inter / best / 1e-3:.3e} interactions/s  counters {list(map(int, cnt))}  "
          f"per target: {cnt[0] / n:.0f} visits {cnt[1] / n:.0f} cells {cnt[2] / n:.0f} pairs")
    if st[3] and st[4]:
        print(f"   lane use: pair-row slots issued {st[3]} (useful {st[2] / st[3]:.3f}), node-visit target slots issued "
              f"{st[4]} (awake {st[5] / st[4]:.3f}; {st[4] / n:.0f} per target)")
    eng.close()


if __name__ == "__main__":
    main()
