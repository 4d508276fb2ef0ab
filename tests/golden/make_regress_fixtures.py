"""Sub-samples the reference's golden trajectories (regress/*.dat, written by programs/regress.cpp:78-95:
`t q0 q1 ...` per step, generalized Euler coordinates of every body) into small fixtures.
Needs the original Moby sources: MOBY_SOURCE_DIR names a Moby checkout.  The fixtures are committed.
"""
import os
import sys
import numpy as np

if not os.environ.get("MOBY_SOURCE_DIR"):
    sys.exit("set MOBY_SOURCE_DIR to a checkout of the original Moby sources (this script reads its regress/*.dat)")
REF = os.path.join(os.environ["MOBY_SOURCE_DIR"], "regress")
OUT = os.path.dirname(os.path.abspath(__file__))


def load(name):
    rows = []
    with open(os.path.join(REF, name)) as f:
        for line in f:
            p = line.split()
            if len(p) > 1:          # the last line is the CPU-seconds timing row (regress.cpp:274-277)
                rows.append([float(x) for x in p])
    return np.array(rows)


for name, every in (("sitting-box.dat", 200), ("sphere-stack.dat", 10), ("rimless-wheel.dat", 50), ("contact-constrained-pendulum.dat", 50)):
    a = load(name)
    idx = sorted(set(list(range(0, 6)) + list(range(0, len(a), every)) + [len(a) - 1]))
    np.savetxt(os.path.join(OUT, "regress_" + name.replace(".dat", ".txt").replace("-", "_")), a[idx], fmt="%.6g",
               header=f"rows {len(idx)} of {len(a)} from {name} (6 significant digits as written by moby-regress)")
    print(name, a.shape, len(idx))
