"""Time of the L-mer table (gkmb200_lmer_table_*, DESIGN.md 4.5) against the fused decision values on the same rows, on one
GPU, for two workloads:
  configs[4] per GPU  125 000 test rows x 300 bp, 10 000 SVs, type 2, L = 11, k = 7, d = 3, bench.py's alpha and bias
  gkmQC's default     wgkm (type 4, M = H = 50), L = 10, k = 6, d = 3, 600-bp windows, same counts
Timed after one warm-up of each call, host clock around synchronised calls, `reps` times each: the table build (and its
three phases S, transform, combine in device time from CUDA events), the scoring of all test rows, and
gkmb200_decision_values over the same rows.  Also the largest |table - decision values| / eps(r) over sampled rows
(eps: tests/test_lmer_table_model.py), and the card's name and power limit.

    python tools/lmer_table_bench.py [reps] [out.json]
"""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
from gkmqc_b200 import capi  # noqa: E402
import bench  # noqa: E402
import lmer_table_model as ltm  # noqa: E402

reps = int(sys.argv[1]) if len(sys.argv) > 1 else 5
out_path = sys.argv[2] if len(sys.argv) > 2 else None
capi.load()
if capi.device_count() < 1:
    raise SystemExit("needs a B200: " + capi.last_error())
import ctypes  # noqa: E402
assert capi.load().gkmb200_set_devices((ctypes.c_int * 1)(0), 1) == 0
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()

NSV, NTEST = bench.NSV, bench.NTEST_PER_GPU
WORKLOADS = [("configs[4] per GPU", dict(kernel_type=2, L=11, k=7, d=3), 300),
             ("gkmQC default (wgkm)", dict(kernel_type=4, L=10, k=6, d=3, M=50, H=50.0), 600)]


def timed(fn):
    fn()  # warm-up
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        r = fn()
        ts.append(time.perf_counter() - t0)
    return r, ts


results = {"gpu": gpu, "reps": reps, "workloads": []}
for name, params, seqlen in WORKLOADS:
    sv = bench.synth(NSV, seed=99, seqlen=seqlen)
    test = bench.synth(NTEST, seed=1000, seqlen=seqlen)
    alpha = np.random.default_rng(3).standard_normal(NSV)
    with capi.Problem(**params) as P:
        P.add_block(sv)
        P.add_block(test)
        P.upload()
        phases = []

        def build():
            t = P.lmer_table(0, NSV, alpha)
            phases.append(t.build_ms())
            return t

        tabs = []
        _, t_build = timed(lambda: tabs.append(build()) or tabs[-1])
        tab = tabs[-1]
        for t in tabs[:-1]:
            t.close()
        scores, t_score = timed(lambda: tab.scores(P, NSV, NTEST, bias=-0.1))
        dv, t_dv = timed(lambda: P.decision_values(NSV, NTEST, 0, NSV, alpha, bias=-0.1))
        # deviation against eps(r) on sampled rows (B from the histograms of those rows)
        pick = np.unique(np.linspace(0, NTEST - 1, 64).astype(int))
        norm = P.sqnorm()
        model = ltm.Model(P, params["kernel_type"], params["L"], params["d"], params.get("M", 50), params.get("H", 50.0))
        run = model.longest_run(0, NSV)
        w = np.abs(model.w)
        worst = 0.0
        for i in pick:
            r = NSV + int(i)
            H = P.hist_block(r, 1, 0, NSV)[0].astype(np.float64)
            B = (H @ w) @ (np.abs(alpha) / norm[:NSV]) / norm[r]
            eps = (NSV + run + 4 * params["L"] + (seqlen - params["L"] + 1) + 16) * 2.0 ** -52 * B
            worst = max(worst, abs(scores[i] - dv[i]) / eps)
        tab.close()
        ph = np.median(np.array(phases[1:]), axis=0)
        rec = {"workload": name, "params": params, "seqlen": seqlen, "nsv": NSV, "ntest": NTEST,
               "build_ms_median": 1e3 * float(np.median(t_build)), "build_device_ms_median": {"S": ph[0], "transform": ph[1], "combine": ph[2]},
               "score_ms_median": 1e3 * float(np.median(t_score)), "decision_values_ms_median": 1e3 * float(np.median(t_dv)),
               "build_ms_all": [1e3 * x for x in t_build], "score_ms_all": [1e3 * x for x in t_score], "dv_ms_all": [1e3 * x for x in t_dv],
               "max_dev_over_eps_sampled": worst, "sampled_rows": int(len(pick)), "longest_run": run}
        results["workloads"].append(rec)
        print(json.dumps(rec), flush=True)
print(json.dumps({"gpu": gpu}))
if out_path:
    with open(out_path, "w") as f:
        json.dump(results, f, indent=1)
