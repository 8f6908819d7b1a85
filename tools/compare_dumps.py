"""Compares two `bench.py --dump-outputs` directories array by array and prints (or writes with --out) one JSON record:
for every array, whether the two builds wrote the same bits and the largest absolute difference.

    python tools/compare_dumps.py DIR_A DIR_B [--label cifar10] [--out result.json]
"""
import argparse
import json
import os

import numpy as np


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("a")
    ap.add_argument("b")
    ap.add_argument("--label", default="")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    names = sorted(f[:-4] for f in os.listdir(args.a) if f.endswith(".npy"))
    if names != sorted(f[:-4] for f in os.listdir(args.b) if f.endswith(".npy")):
        raise SystemExit("the two directories hold different arrays")
    rec = {"label": args.label, "arrays": {}}
    for n in names:
        x, y = np.load(os.path.join(args.a, n + ".npy")), np.load(os.path.join(args.b, n + ".npy"))
        same = x.shape == y.shape and x.dtype == y.dtype and x.tobytes() == y.tobytes()
        diff = float(np.abs(x.astype(np.float64) - y.astype(np.float64)).max()) if x.shape == y.shape else None
        rec["arrays"][n] = {"shape": list(x.shape), "bit_identical": same, "max_abs_diff": diff}
    rec["all_bit_identical"] = all(v["bit_identical"] for v in rec["arrays"].values())
    doc = json.dumps(rec, indent=1)
    print(doc)
    if args.out:
        with open(args.out, "w") as f:
            f.write(doc + "\n")


if __name__ == "__main__":
    main()
