"""Time of the single-base substitutions (gkmb200_lmer_table_substitutions, DESIGN.md 4.6) on one GPU, against gkmQC's default
model (wgkm, type 4, M = H = 50, L = 10, k = 6, d = 3) folded from 10 000 SVs of 600 bp:
  (a) full ISM of 10 000 x 600-bp rows (6 M sites, 24 M scores)
  (b) 100 000 one-site 600-bp rows (the variant-effect shape)
  (c) 200 rows sampled from (a), full ISM: the new entry point against materialise-and-score (add the 3 x 600 x 4 mutant
      sequences to a new problem, upload it with its sqnorm, LmerTable.scores), both outputs compared bit for bit
Timed with a host clock around synchronised calls after one warm-up, `reps` times each, median; the card's name and power
limit are read in the same run.

    python tools/lmer_subst_bench.py [reps] [out.json]
"""
import ctypes
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from gkmqc_b200 import capi  # noqa: E402
import bench  # noqa: E402

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
out_path = sys.argv[2] if len(sys.argv) > 2 else None
capi.load()
if capi.device_count() < 1:
    raise SystemExit("needs a B200: " + capi.last_error())
assert capi.load().gkmb200_set_devices((ctypes.c_int * 1)(0), 1) == 0
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()

PARAMS = dict(kernel_type=4, L=10, k=6, d=3, M=50, H=50.0)
NSV, NROWS, NVAR, NSUB, LEN = 10000, 10000, 100000, 200, 600


def timed(fn):
    r = fn()  # warm-up
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        r = fn()
        ts.append(time.perf_counter() - t0)
    return r, ts


def rec(name, sites, ts, **kw):
    med = float(np.median(ts))
    r = {"workload": name, "sites": int(sites), "ms_median": 1e3 * med, "sites_per_s": sites / med, "ms_all": [1e3 * x for x in ts]}
    r.update(kw)
    print(json.dumps(r), flush=True)
    return r


results = {"gpu": gpu, "reps": reps, "params": PARAMS, "nsv": NSV, "seqlen": LEN, "workloads": []}
sv = bench.synth(NSV, seed=99, seqlen=LEN)
alpha = np.random.default_rng(3).standard_normal(NSV)
with capi.Problem(**PARAMS) as S:
    S.add_block(sv)
    tab = S.lmer_table(0, NSV, alpha)
    with capi.Problem(**PARAMS) as P:  # (a)
        rows_a = bench.synth(NROWS, seed=1000, seqlen=LEN)
        P.add_block(rows_a)
        P.upload()
        rows = np.repeat(np.arange(NROWS, dtype=np.int32), LEN)
        pos = np.tile(np.arange(LEN, dtype=np.int32), NROWS)
        ism, ts = timed(lambda: tab.substitutions(P, rows, pos, bias=-0.1))
        results["workloads"].append(rec("(a) full ISM, 10 000 x 600 bp", len(rows), ts))
        # (c) 200 rows of (a): the entry point against materialise-and-score
        pick = np.arange(0, NROWS, NROWS // NSUB)[:NSUB]
        r_c = np.repeat(pick.astype(np.int32), LEN)
        p_c = np.tile(np.arange(LEN, dtype=np.int32), NSUB)
        sub, ts_new = timed(lambda: tab.substitutions(P, r_c, p_c, bias=-0.1))
        mut = np.repeat(rows_a[pick], 4 * LEN, axis=0).reshape(NSUB, LEN, 4, LEN)
        for v in range(4):
            mut[:, np.arange(LEN), v, np.arange(LEN)] = bench.ACGT[v]
        mut = mut.reshape(-1, LEN)

        def materialise():
            with capi.Problem(**PARAMS) as Q:
                Q.add_block(mut)
                Q.upload()
                return tab.scores(Q, 0, Q.n, bias=-0.1)

        mat, ts_mat = timed(materialise)
        same = bool(np.array_equal(sub.reshape(-1).view(np.uint64), mat.view(np.uint64)))
        same_a = bool(np.array_equal(ism.reshape(NROWS, LEN, 4)[pick].reshape(-1).view(np.uint64), mat.view(np.uint64)))
        results["workloads"].append(rec("(c) 200 x 600 bp, substitutions", len(r_c), ts_new))
        results["workloads"].append(rec("(c) 200 x 600 bp, materialise + upload + scores", len(r_c), ts_mat,
                                        mutant_sequences=int(len(mut)), bit_identical=same, bit_identical_to_a=same_a))
        assert same and same_a, "substitutions differ from the materialised mutants"
    with capi.Problem(**PARAMS) as V:  # (b)
        V.add_block(bench.synth(NVAR, seed=2000, seqlen=LEN))
        V.upload()
        pos_b = np.random.default_rng(5).integers(0, LEN, NVAR).astype(np.int32)
        _, ts = timed(lambda: tab.substitutions(V, np.arange(NVAR, dtype=np.int32), pos_b, bias=-0.1))
        results["workloads"].append(rec("(b) 100 000 one-site rows, 600 bp", NVAR, ts))
    tab.close()
print(json.dumps({"gpu": gpu}))
if out_path:
    with open(out_path, "w") as f:
        json.dump(results, f, indent=1)
