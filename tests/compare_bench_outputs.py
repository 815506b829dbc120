"""Run-to-run spread of `bench.py --dump-outputs` against the difference between two builds.

    python tests/compare_bench_outputs.py A1 A2 ... -- B1 B2 ...

Each argument is a directory written by `bench.py --dump-outputs`.  The base preset's training step is not bit-reproducible (the hash-table
gradients are summed with red.global reductions in whatever order the warps reach them, and Adam's first steps amplify the last bits of
near-zero gradients), so two runs of the SAME build differ.  For every dumped array this prints the largest and median difference between runs
of build A, between runs of build B, and across the builds: a change that computes what its parent computes shows cross-build differences
inside the within-build spread.  It also prints, per build, the mean and standard deviation of every scalar and of every array's RMS
distance to the first run of A (that run itself left out): the two builds' distributions should coincide."""
import itertools
import os
import sys

import numpy as np


def distances(x, y):
    d = np.abs(x.astype(np.float64) - y.astype(np.float64))
    return float(d.max()) if d.size else 0.0, float(np.sqrt((d * d).mean())) if d.size else 0.0


def main():
    args = sys.argv[1:]
    if "--" not in args:
        raise SystemExit(__doc__)
    k = args.index("--")
    A, B = args[:k], args[k + 1:]
    names = sorted(f for f in os.listdir(A[0]) if f.endswith(".npy"))
    load = lambda d, f: np.load(os.path.join(d, f))  # noqa: E731
    print(f"{'array':32s} {'within A max|d| (rms)':>26s} {'within B max|d| (rms)':>26s} {'A vs B max|d| (rms)':>26s}")
    for f in names:
        cols = []
        for pairs in (itertools.combinations(A, 2), itertools.combinations(B, 2), itertools.product(A, B)):
            ds = [distances(load(a, f), load(b, f)) for a, b in pairs]
            cols.append(f"{max(m for m, _ in ds):.3e} ({max(r for _, r in ds):.2e})" if ds else "-")
        print(f"{f[:-4]:32s} {cols[0]:>26s} {cols[1]:>26s} {cols[2]:>26s}")
    print(f"\n{'array':32s} {'A: mean +- std (n)':>36s} {'B: mean +- std (n)':>36s}   (scalars: value; arrays: rms distance to " + A[0] + ")")
    for f in names:
        ref = load(A[0], f)
        cols = []
        for runs in (A[1:] if ref.size > 1 else A, B):
            v = np.array([load(d, f).item() if ref.size == 1 else distances(load(d, f), ref)[1] for d in runs], dtype=np.float64)
            cols.append(f"{v.mean():.6e} +- {v.std(ddof=1) if v.size > 1 else 0.0:.2e} ({v.size})")
        print(f"{f[:-4]:32s} {cols[0]:>36s} {cols[1]:>36s}")


if __name__ == "__main__":
    main()
