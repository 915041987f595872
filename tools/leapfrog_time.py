"""Times leapfrog_kernel (fused kick-kick-drift) at n particles with CUDA events: 68 B per particle against the
measured HBM copy bandwidth."""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, os.path.join(ROOT, "lambda-cdm-raytracing_b200", "python"))


def main():
    import torch
    import torch.distributed as dist
    import b200grav
    import bench
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=1 << 24)
    args = ap.parse_args()
    torch.cuda.set_device(0)
    eng = b200grav.Engine(0)
    D = bench.Dist(torch, dist, 1, 0, torch.device("cuda", 0))
    out = bench.leapfrog_roofline(eng, D, args.n)
    print(json.dumps(out))
    eng.close()


if __name__ == "__main__":
    main()
