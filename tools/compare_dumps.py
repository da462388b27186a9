"""Compare two `bench.py --dump-outputs` directories: every array bit for bit, except `st_sum` (an atomics-ordered
float64 sum) to 1e-6 relative, as bench's parity does.
usage: python tools/compare_dumps.py DIR_A DIR_B"""
import os
import sys

import numpy as np

a_dir, b_dir = sys.argv[1], sys.argv[2]
names = sorted(f for f in os.listdir(a_dir) if f.endswith(".npy"))
assert names == sorted(f for f in os.listdir(b_dir) if f.endswith(".npy")), "different array sets"
bad = 0
for f in names:
    a, b = np.load(os.path.join(a_dir, f)), np.load(os.path.join(b_dir, f))
    if f == "st_sum.npy":
        ok = a.shape == b.shape and np.allclose(a, b, rtol=1e-6, atol=0, equal_nan=True)
    else:
        ok = a.shape == b.shape and a.dtype == b.dtype and np.array_equal(a, b, equal_nan=True)
    print("%-20s %-9s %s" % (f[:-4], "equal" if ok else "DIFFERS", a.shape))
    bad += not ok
print("all equal" if not bad else "%d arrays differ" % bad)
sys.exit(1 if bad else 0)
