"""Wall time of gkmQC's 50 fits of one 10k bin (5-fold x 10 repeats, C = 1, eps = 1e-3) on the resident matrix, with
and without libsvm's shrinking heuristic (gkmb200_svm_cv_ex), alternating the two; plus iterations, smallest active set,
unshrinks and gradient reconstructions of the shrinking fits.  Same bin as tools/svm_bench.py.

    python tools/svm_shrink_bench.py [n] [reps] [out.json]
"""
import json
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from gkmqc_b200 import capi  # noqa: E402
import bench  # noqa: E402
from sklearn.model_selection import StratifiedKFold  # noqa: E402

n = int(sys.argv[1]) if len(sys.argv) > 1 else 10000
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 5
out = sys.argv[3] if len(sys.argv) > 3 else None
capi.load()
rng = np.random.default_rng(7)
arr = bench.synth(n)
npos = n // 2
motifs = [b"GATAAGGCAT", b"TTGACGTCAA", b"CCCGCCCCTA"]
for i in range(npos):   # plant degenerate motifs in the positives, as tools/svm_bench.py
    for m in motifs[: 1 + i % 3]:
        p = int(rng.integers(0, 290))
        mm = bytearray(m)
        if rng.random() < 0.5:
            mm[int(rng.integers(0, 10))] = b"ACGT"[int(rng.integers(0, 4))]
        arr[i, p:p + 10] = np.frombuffer(bytes(mm), np.uint8)
y = np.concatenate((np.ones(npos, int), np.zeros(n - npos, int)))
splits = []
for r in range(10):
    splits.extend(StratifiedKFold(n_splits=5, shuffle=True, random_state=100 + r).split(np.zeros(n), y))
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                     stdout=subprocess.PIPE, text=True).stdout.strip()
res = {"n": n, "fits": len(splits), "C": 1.0, "eps": 1e-3, "gpu": gpu, "reps": reps}
with capi.Problem(4, 10, 6, 3, 50, 50.0, 1.0) as P:   # gkmQC's defaults: wgkm, L=10 k=6 d=3
    P.add_many([a.tobytes().decode() for a in arr])
    P.resident_matrix(0, 0)
    times = {0: [], 1: []}
    outs = {}
    for shrinking in (0, 1):   # warm-up of both kernels
        capi.svm_cv(y, splits, problem=P, C=1.0, eps=1e-3, shrinking=shrinking, stats=True)
    for _ in range(reps):
        for shrinking in (0, 1):
            t0 = time.perf_counter()
            outs[shrinking] = capi.svm_cv(y, splits, problem=P, C=1.0, eps=1e-3, shrinking=shrinking, stats=True)
            times[shrinking].append(time.perf_counter() - t0)
for shrinking, key in ((0, "no_shrinking"), (1, "shrinking")):
    scores, fits, _, st = outs[shrinking]
    it = [f["n_iter"] for f in fits]
    res[key] = {
        "wall_s_each": times[shrinking], "wall_s_median": float(np.median(times[shrinking])),
        "iters_mean": float(np.mean(it)), "iters_max": int(max(it)),
        "n_sv_mean": float(np.mean([f["n_sv"] for f in fits])),
        "min_active_mean": float(np.mean([s["min_active"] for s in st])), "min_active_min": int(min(s["min_active"] for s in st)),
        "shrink_passes_mean": float(np.mean([s["shrink_passes"] for s in st])),
        "unshrinks": int(sum(s["unshrink_iter"] >= 0 for s in st)),
        "recon_a": int(sum(s["recon_a"] for s in st)), "recon_b": int(sum(s["recon_b"] for s in st)),
    }
    print("%-12s %.3f s median of %d (%s), iterations %.0f mean / %d max, smallest active set %d, reconstructions A %d B %d"
          % (key, res[key]["wall_s_median"], reps, " ".join("%.3f" % t for t in times[shrinking]), res[key]["iters_mean"],
             res[key]["iters_max"], res[key]["min_active_min"], res[key]["recon_a"], res[key]["recon_b"]), flush=True)
d = max(float(np.max(np.abs(a - b))) for a, b in zip(outs[0][0], outs[1][0]))
res["max_abs_diff_decision_values_between_the_two"] = d
print("GPU %s; max |decision value difference| between the two paths %.3g" % (gpu, d))
if out:
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    json.dump(res, open(out, "w"), indent=1)
