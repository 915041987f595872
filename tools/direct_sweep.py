"""Tuning harness for the direct-sum kernel: times every register-blocking
variant (B200_DIRECT_VARIANT = "R,THREADS,MINB") with CUDA events on one problem size and
prints interactions/s and the fraction of the measured FP32 peak."""
import argparse
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "lambda-cdm-raytracing_b200", "python"))


def main():
    import torch
    import b200grav
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=262144)
    ap.add_argument("--variants", default="default;2,256,2;4,256,1;4,256,2;5,256,1;6,256,1;7,256,1;8,256,1;4,384,1;4,512,1;3,512,1;6,128,2;8,128,2")
    ap.add_argument("--masses", default="unit", choices=["unit", "random"])
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--box", type=float, default=0.0, help="> 0: the periodic (minimum-image) instance")
    args = ap.parse_args()
    eng = b200grav.Engine(0)
    rng = np.random.default_rng(0)
    n = args.n
    mass = np.ones((n, 1)) if args.masses == "unit" else rng.uniform(0.5, 1.5, (n, 1))
    posm = torch.from_numpy(np.concatenate([rng.uniform(-50, 50, (n, 3)), mass], 1).astype(np.float32)).cuda()
    acc = torch.empty((n, 3), dtype=torch.float32, device="cuda")
    peak = max(eng.fp32_peak_probe(0, 4000)[0], eng.fp32_peak_probe(1, 4000)[0])
    print(f"n={n} masses={args.masses} fp32 peak (probe) {peak:.2f} TFLOP/s")
    eng.set_timing(True)
    ref = None
    for v in args.variants.split(";"):
        # periodic only: a "float:" prefix picks the FP32 minimum image (default: fixed point)
        os.environ.pop("B200_DIRECT_PERIODIC_FLOAT", None)
        label = v
        if v.startswith("float:"):
            os.environ["B200_DIRECT_PERIODIC_FLOAT"] = "1"; v = v[6:]
        if v.startswith("default"):
            os.environ.pop("B200_DIRECT_VARIANT", None)
            v = "default"
        else:
            os.environ["B200_DIRECT_VARIANT"] = v
        best = 1e30
        for _ in range(args.reps):
            eng.direct_forces_dev(posm, acc, 0, n, eps=0.01, box=args.box)
            torch.cuda.synchronize()
            best = min(best, eng.last_kernel_ms())
        a = acc.cpu().numpy()
        if ref is None:
            ref = a
        err = float(np.sqrt(((a - ref) ** 2).sum() / (ref ** 2).sum()))
        rate = float(n) * n / (best * 1e-3)
        print(f"variant {label:16s} kernel {best:9.3f} ms  {rate:.4e} int/s  {20 * rate / 1e12:6.2f} TFLOP/s  "
              f"{20 * rate / 1e12 / peak:6.3f} of peak   rel diff vs first {err:.1e}")
    eng.close()


if __name__ == "__main__":
    main()
