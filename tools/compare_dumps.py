"""Compare two `bench.py --dump-outputs` directories: layer samples and step result exactly (or within a relative
tolerance), weight gradients within rtol / atol of their max (atomic accumulation order varies between runs)."""
import argparse
import os
import sys

import numpy as np


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("a")
    ap.add_argument("b")
    ap.add_argument("--rtol", type=float, default=0.0, help="per-element tolerance of samples: rtol*|a| + rtol*rms(a)")
    ap.add_argument("--wg-rtol", type=float, default=2e-2)
    ap.add_argument("--wg-atol", type=float, default=1e-2, help="times max |weight grad|")
    args = ap.parse_args()
    names = sorted(os.listdir(args.a))
    assert names == sorted(os.listdir(args.b)), "different file sets"
    bad = 0
    for n in names:
        x, y = np.load(os.path.join(args.a, n)), np.load(os.path.join(args.b, n))
        if n == "weight_grads.npy":
            ok = np.allclose(y, x, rtol=args.wg_rtol, atol=args.wg_atol * np.abs(x).max())
        elif args.rtol == 0:
            ok = np.array_equal(x, y)
        else:
            rms = float(np.sqrt(np.mean(x.astype(np.float64) ** 2)))
            ok = bool(np.all(np.abs(y - x) <= args.rtol * np.abs(x) + args.rtol * rms))
        rel = float(np.abs(y - x).max() / max(np.abs(x).max(), 1e-30))
        print("%-40s %s  max|diff|/max|a| %.3g" % (n, "ok" if ok else "DIFFERENT", rel))
        bad += not ok
    print("ALL MATCH" if not bad else "%d DIFFER" % bad)
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
