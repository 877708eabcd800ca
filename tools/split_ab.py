#!/usr/bin/env python
"""A/B of how a lower triangle's columns are cut into index blocks (option index_split): equal shares against full blocks
first.  Resident passes at several problem sizes; at 20k also checks that both splits return the same bits.
   python tools/split_ab.py [n ...]      (default 20000 28288 50000)"""
import json
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench
from gkmqc_b200 import capi

sizes = [int(a) for a in sys.argv[1:]] or [20000, 28288, 50000]
res = {}


def timed(n, split, cols=0, kt=2, L=11, k=7, d=3):
    capi.set_option("index_split", split)
    capi.set_option("index_cols", cols)
    with capi.Problem(kt, L, k, d) as P:
        P.add_block(bench.synth(n))
        ms = P.bench_lower_resident(2, 1, True)
        out = {"ms": float(ms.mean()), "launches": P.stats()["launches"], "layout": P.index_layout()}
    key = "n%d_t%d_%s_cols%d" % (n, kt, split, cols)
    res[key] = out
    print(key, out, flush=True)
    with open("gpurun_out/split_ab.json", "w") as f:
        json.dump(res, f, indent=1)
    return out


os.makedirs("gpurun_out", exist_ok=True)
capi.set_option("kernel", "index")
# the same bits from both splits: rows on both sides of the block boundaries of either layout, dense and histograms
n = 20000
rows = [1, 2, 10015, 10016, 10017, 16383, 16384, 16385, 19998, 19999]
got = {}
for split in ("equal", "greedy"):
    capi.set_option("index_split", split)
    with capi.Problem(2, 11, 7, 3) as P:
        P.add_block(bench.synth(n))
        got[split] = [(P.kernel_block(r, 1, 0, n, lower=True).copy(), P.hist_block(r, 1, 0, n, lower=True).copy()) for r in rows]
        print(split, "layout", P.index_layout(), flush=True)
same = all(np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]) for a, b in zip(got["equal"], got["greedy"]))
print("same bits from both splits at %d rows of 20k: %s" % (len(rows), same), flush=True)
res["same_bits_20k"] = bool(same)

for n in sizes:
    timed(n, "equal")
    timed(n, "greedy")
    if n >= 40000:
        timed(n, "greedy", cols=14336)
# gkmQC's weighted default kernel type at 20k x 300 bp (two blocks either way; W20 slots hold 16 352 columns at most)
timed(20000, "equal", kt=4, L=10, k=6, d=3)
timed(20000, "greedy", kt=4, L=10, k=6, d=3)
