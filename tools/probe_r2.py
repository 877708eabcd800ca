#!/usr/bin/env python
"""Round-2 measurement session on one box (writes gpurun_out/probe_r2.json + .log):
   micro-benchmarks, anatomy of the end-to-end call at 50k / 10k under copy-thread and huge-page settings,
   gkmQC's default configuration (wgkm L=10 k=6 d=3, 600 bp), d = 4, kernel variants.
   python tools/probe_r2.py [what ...]      what in: micro e2e50 e2e10 default d4 variants"""
import json, os, subprocess, sys, tempfile, time
import numpy as np
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench
from gkmqc_b200 import capi

what = sys.argv[1:] or ["micro", "e2e50", "e2e10", "default", "d4"]
out_dir = os.path.join(ROOT, "gpurun_out")
os.makedirs(out_dir, exist_ok=True)
res = {"cores": len(os.sched_getaffinity(0)), "thp": bench.thp_mode(), "devices": capi.device_count()}
tmp = tempfile.mkdtemp(dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
lib = capi.load()


def save():
    json.dump(res, open(os.path.join(out_dir, "probe_r2.json"), "w"), indent=1)


def resident(ktype, L, k, d, arr, kernel="auto", steps=2, **kw):
    capi.set_option("kernel", kernel)
    try:
        with capi.Problem(ktype, L, k, d, **kw) as P:
            P.add_block(arr)
            ms = P.bench_lower_resident(steps, 1, True)
            st = P.stats()
            return {"ms": float(ms.mean()), "variant": bench.VARIANTS.get(st["kernel_variant"]), "layout": P.index_layout(),
                    "M_entries_s": len(arr) * (len(arr) - 1) / 2 / ms.mean() / 1e3}
    finally:
        capi.set_option("kernel", "auto")


if "micro" in what:
    res["micro"] = {w: capi.microbench(w) for w in ("gather16", "atoms7", "atoms32", "lop3", "popc")}
    print(res["micro"], flush=True); save()

def e2e(n, tag, env=None, reps=3, seqlen=300, **kw):
    pos, neg = bench.write_problem(tmp, n, seqlen=seqlen, tag="_%s" % tag)
    old = {}
    for k_, v_ in (env or {}).items():
        old[k_] = os.environ.get(k_)
        os.environ[k_] = v_
    walls, stats = [], None
    try:
        for it in range(reps + 1):
            km = np.zeros((n, n))
            t0 = time.perf_counter()
            ret, km, a, b = capi.main_pywrapper(pos, neg, nthreads=1, verbosity=3 if it == reps else 0, kmat=km, **kw)
            w = time.perf_counter() - t0
            assert ret == 0, capi.last_error()
            st = capi.gkmb200_stats(); lib.gkmb200_get_stats(None, capi.ctypes.byref(st))
            stats = st.as_dict()
            walls.append(w)
            t0 = time.perf_counter(); del km; tfree = time.perf_counter() - t0
    finally:
        for k_, v_ in old.items():
            if v_ is None: os.environ.pop(k_, None)
            else: os.environ[k_] = v_
    return {"n": n, "env": env, "walls_s": walls, "stats": stats, "free_s": tfree}

if "e2e50" in what:
    res["e2e50"] = {}
    for tag, env in (("default", {}), ("threads8", {"GKM_COPY_THREADS": "8"}), ("threads16", {"GKM_COPY_THREADS": "16"}),
                     ("threads32", {"GKM_COPY_THREADS": "32"})):
        res["e2e50"][tag] = e2e(50000, "50k", env, reps=2, kernel_type=2, L=11, k=7, d=3)
        print(tag, res["e2e50"][tag]["walls_s"], res["e2e50"][tag]["stats"], flush=True); save()

if "e2e10" in what:
    res["e2e10"] = {}
    for tag, env in (("default", {}), ("threads8", {"GKM_COPY_THREADS": "8"})):
        res["e2e10"][tag] = e2e(10000, "10k", env, reps=3, kernel_type=2, L=11, k=7, d=3)
        print(tag, res["e2e10"][tag]["walls_s"], res["e2e10"][tag]["stats"], flush=True); save()

if "default" in what:
    res["default"] = {}
    a600 = bench.synth(10000, seed=4321, seqlen=600)
    a300 = bench.synth(10000)
    for tag, arr, args in (("t4_L10_600bp", a600, (4, 10, 6, 3)), ("t2_L10_600bp", a600, (2, 10, 6, 3)), ("t4_L10_300bp", a300, (4, 10, 6, 3)),
                           ("t4_L11_300bp", a300, (4, 11, 7, 3)), ("t2_L11_300bp", a300, (2, 11, 7, 3)), ("t2_L11_600bp", a600, (2, 11, 7, 3))):
        for kern in ("index", "diag"):
            if kern == "diag" and tag not in ("t4_L10_600bp", "t2_L11_300bp"):
                continue
            res["default"]["%s_%s" % (tag, kern)] = resident(*args, arr, kernel=kern)
            print(tag, kern, res["default"]["%s_%s" % (tag, kern)], flush=True); save()
    for cols in (2048, 4096, 6144):
        capi.set_option("index_cols", cols)
        res["default"]["t4_L10_600bp_index_cols%d" % cols] = resident(4, 10, 6, 3, a600, kernel="index")
        print(cols, res["default"]["t4_L10_600bp_index_cols%d" % cols], flush=True); save()
    capi.set_option("index_cols", 0)

if "d4" in what:
    res["d4"] = {}
    a20 = bench.synth(20000)
    for tag, args in (("L11_d4", (2, 11, 7, 4)), ("L11_d3", (2, 11, 7, 3)), ("L10_d4", (2, 10, 6, 4)), ("L12_d4", (2, 12, 8, 4))):
        res["d4"][tag] = resident(*args, a20, kernel="index", steps=1)
        print(tag, res["d4"][tag], flush=True); save()

if "blocks50" in what:
    res["blocks50"] = {}
    a50 = bench.synth(50000)
    for cols in (0, 10016, 8352, 16384):
        capi.set_option("index_cols", cols)
        res["blocks50"]["cols%d" % cols] = resident(2, 11, 7, 3, a50, kernel="index", steps=1)
        print(cols, res["blocks50"]["cols%d" % cols], flush=True); save()
    capi.set_option("index_cols", 0)

if "variants" in what:
    res["variants"] = {}
    a = bench.synth(4000)
    for kern in ("index", "diag", "mma", "lmer"):
        res["variants"][kern] = resident(2, 11, 7, 3, a, kernel=kern, steps=1)
        print(kern, res["variants"][kern], flush=True); save()
save()

save()
