#!/usr/bin/env python
"""bench.py -- gkm kernel entries/s (300 bp, L=11 k=7 d=3) on N B200s, next to the reference's CPU path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One process per GPU (torchrun sets RANK/LOCAL_RANK/WORLD_SIZE); torch.distributed is used for the barrier and the
max-over-ranks only -- the path has no collective.  A "step" is one full pass of the hot path: the strict lower
triangle of the kernel matrix of the workload below.

Workload (BASELINE.json configs[3], the north-star target): 25 000 + 25 000 synthetic 300-bp sequences, the full
50k x 50k kernel matrix, kernel type 2 (EST_TRUNC), L=11 k=7 d=3 -- the SAME problem at every N ("scaling": "strong"):
its chunks of row tiles are sharded round-robin over the ranks.

  value     device-resident: packed sequences and the output matrix stay in HBM, CUDA-event time of the pass
  e2e       gkm_main_pywrapper(FASTA files -> caller's fresh numpy rows), wall clock: file parse, pack, H2D, sqnorm,
            index build, kernels, D2H and the copy into the caller's matrix all inside the timed region
  parity    rows of the matrix the e2e call RETURNED (and their integer histograms through gkmb200_hist_block)
            against the unmodified reference (oracle/_ref) -- a mismatch makes the run exit non-zero
  secondary configs[1] (10k, resident + e2e + one full unsampled run of the reference's own gkm_main_pywrapper),
            gkmQC's real default (wgkm L=10 k=6 d=3 on 600-bp sequences), non-uniform input, configs[4] batch scoring

--dump-outputs DIR writes what the last timed e2e call returned to its caller (the resident pass behind `value` keeps its
matrix on the device and returns nothing): a seeded sample of the rows rank 0 filled, their row ids and (npos, nneg).
"""
import argparse
import ctypes
import hashlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

L, K, D, KTYPE, SEQLEN = 11, 7, 3, 2, 300
BASE_N = 50000          # BASELINE.json configs[3]
SECOND_N = 10000        # BASELINE.json configs[1]
NSV, NTEST_PER_GPU = 10000, 125000   # BASELINE.json configs[4]: 1M test x 10k SV over 8 GPUs = 125k test rows per GPU
PAIRS_PER_ENTRY = (SEQLEN - L + 1) * 2 * (SEQLEN - L + 1)   # 168 200 L-mer pair comparisons (SURVEY.md 8d)
INT_OPS_PER_PAIR = 5                                        # canonical XOR/SHR/LOP3/POPC/ISETP count (SURVEY.md 8d)
METRIC = "gkm kernel entries/sec (300bp, l=11 k=7 d=3)"
VARIANTS = {1: "lmer", 2: "diag", 3: "mma", 4: "index"}
ACGT = np.frombuffer(b"ACGT", dtype=np.uint8)


def synth(n, seed=1234, seqlen=SEQLEN):
    rng = np.random.default_rng(seed)
    return ACGT[rng.integers(0, 4, size=(n, seqlen))]


def write_fasta(path, arr, first_id):
    """>s<i>\\n<bases>\\n per row, assembled in numpy (50k records in ~50 ms)"""
    n, ln = arr.shape
    ids = [b">s%d\n" % i for i in range(first_id, first_id + n)]
    with open(path, "wb") as f:
        rows = [None] * (2 * n)
        rows[0::2] = ids
        body = np.concatenate((arr, np.full((n, 1), 10, np.uint8)), axis=1)
        rows[1::2] = [body[i].tobytes() for i in range(n)]
        f.write(b"".join(rows))


def write_problem(tmp, n, seed=1234, seqlen=SEQLEN, tag=""):
    arr = synth(n, seed, seqlen)
    half = n // 2
    pos, neg = os.path.join(tmp, "pos%s.fa" % tag), os.path.join(tmp, "neg%s.fa" % tag)
    write_fasta(pos, arr[:half], 0)
    write_fasta(neg, arr[half:], half)
    return pos, neg


class ClockSampler(threading.Thread):
    """nvidia-smi clocks and throttle reasons during the timed region (B200_PROFILING.md)"""

    def __init__(self, gpu):
        super().__init__(daemon=True)
        self.gpu = gpu
        self.rows = []
        self.stop_flag = False
        self.proc = None

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                self.rows.append([x.strip() for x in line.split(",")])
                if self.stop_flag:
                    break
        except Exception:
            pass

    def finish(self):
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        sm, reasons = [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0]))
                out["sm_max_mhz"] = float(r[1])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            except (ValueError, IndexError):
                continue
        if sm:
            top = sorted(sm)[len(sm) // 2:]   # samples under load: the upper half
            out["sm_mhz"] = float(np.median(top))
        out["reasons"] = sorted(reasons)
        out["samples"] = len(sm)
        return out


def dist_setup(world):
    if world <= 1:
        return None
    import torch
    import torch.distributed as dist
    os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
    backend = "nccl" if torch.cuda.is_available() else "gloo"
    if backend == "nccl":
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", "0")))
    # NCCL prints its version banner on stdout when the first communicator comes up; stdout carries the
    # one JSON line only, so that banner goes to stderr
    sys.stdout.flush()
    saved = os.dup(1)
    os.dup2(2, 1)
    try:
        dist.init_process_group(backend=backend)
        dev = "cuda" if backend == "nccl" else "cpu"
        t = torch.zeros(1, device=dev)
        dist.all_reduce(t)
        if backend == "nccl":
            torch.cuda.synchronize()
    finally:
        sys.stdout.flush()
        os.dup2(saved, 1)
        os.close(saved)
    return dist


def _dist_reduce(dist, x, op):
    if dist is None:
        return x
    import torch
    dev = "cuda" if dist.get_backend() == "nccl" else "cpu"
    t = torch.tensor([x], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=getattr(dist.ReduceOp, op))
    return float(t.item())


def dist_max(dist, x):
    return _dist_reduce(dist, x, "MAX")


def dist_sum(dist, x):
    return _dist_reduce(dist, x, "SUM")


def dist_barrier(dist):
    if dist is not None:
        dist.barrier()


def index_probe_counts(L_, d_, slot_bytes):
    """probes and distinct 32-byte sectors per query L-mer of the index variant, from the product's own mask list
    (slot_bytes = 8: compact slots, 16: wide slots with weights)"""
    from gkmqc_b200 import capi
    lib = capi.load()
    lib.gkm_idx_delta_count.restype = ctypes.c_longlong
    lib.gkm_idx_deltas.restype = ctypes.c_longlong
    lib.gkm_idx_deltas.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_longlong]
    nd = lib.gkm_idx_delta_count(L_, d_)
    a = np.zeros(nd, dtype=np.uint32)
    assert lib.gkm_idx_deltas(L_, d_, a.ctypes.data, nd) == nd
    return int(nd), int(len(np.unique((a & 0x0FFFFFFF) >> (2 if slot_bytes == 8 else 1))))   # 32-byte sector = 4 or 2 slots


def measured_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def kernel_source_hash():
    """identity of the dominant kernel's source: an ncu capture is only attached to a bench line of the same code"""
    h = hashlib.sha256()
    for f in ("gkm_index.cu", "gkm_index.h", "gkm_index_dev.h"):
        h.update(open(os.path.join(ROOT, "gkmqc_b200", "csrc", f), "rb").read())
    return h.hexdigest()[:16]


def thp_mode():
    try:
        return open("/sys/kernel/mm/transparent_hugepage/enabled").read().strip()
    except Exception:
        return None


# ---------------------------------------------------------------------------------------- the reference on the CPU
def open_reference(pos, neg, ktype=KTYPE, L_=L, k_=K, d_=D):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pyoracle
    if not pyoracle.have_ref():
        return None
    t0 = time.time()
    h = pyoracle.RefHook(pos, neg, ktype, L_, k_, d_)
    h.open_s = time.time() - t0
    return h


def reference_rate(h, n, budget_s, threads, endcap=0):
    """the reference's own row loop (oracle/_ref, unmodified sources) on evenly spaced rows of the OPEN problem (k-mer
    tree over all of its sequences), sized to about budget_s seconds"""
    cost = (lambda rows: float(len(rows)) * endcap) if endcap else (lambda rows: float(rows.sum()))
    lo = n // 4 if not endcap else endcap
    probe = np.linspace(lo, n - 1, 2 * threads).astype(np.int32)
    t, _ = h.rows_timed(probe, threads, endcap)
    rate = cost(probe) / max(t, 1e-9)
    per_row = (n / 2.0) if not endcap else float(endcap)
    nrows = int(min(n - 1 - (endcap or 0), max(threads, rate * budget_s / per_row)))
    rows = np.unique(np.linspace(1 if not endcap else endcap, n - 1, nrows).astype(np.int32))
    t, _ = h.rows_timed(rows, threads, endcap)
    entries = cost(rows)
    return dict(value=entries / t, unit="entries/s", cores=threads, kind="reference",
                sample="%d evenly spaced rows of the %d-sequence problem (%d entries, %.1f s on %d threads), k-mer tree over all sequences"
                       % (len(rows), n, int(entries), t, threads))


def port_rate(pos, neg, n):
    """fallback where the reference was not built: the brute-force oracle port"""
    import pyoracle
    o = pyoracle.Oracle(KTYPE, L, K, D)
    o.read_problem(pos, neg)
    rows = np.linspace(1, n - 1, 4).astype(np.int32)
    t0 = time.time()
    o.rect(rows, 256, with_hist=False)
    t = time.time() - t0
    return dict(value=len(rows) * 256 / t, unit="entries/s", cores=1, kind="port",
                sample="%d rows x 256 columns by the brute-force oracle port (%.1f s)" % (len(rows), t))


def parity_rows(n, blk_cols, nblk, want=96, seed=7):
    """rows 1 and n-1, both sides of every column-block boundary of the index, both sides of chunk boundaries
    (multiples of 148 rows: one CTA per SM and wave; chunks hold up to 4 waves) spread over the matrix, random rows"""
    rows = {1, 2, n - 2, n - 1}
    for k in range(1, max(nblk, 1)):
        cb = k * blk_cols
        rows.update(r for r in (cb - 1, cb, cb + 1) if 0 < r < n)
    waves = np.unique(np.linspace(1, (n - 1) // 148, 14).astype(int))
    for w in waves:
        rows.update(r for r in (148 * w - 1, 148 * w) if 0 < r < n)
    for w in np.unique(np.linspace(1, (n - 1) // 592, 6).astype(int)):
        rows.update(r for r in (592 * w - 1, 592 * w) if 0 < r < n)
    rng = np.random.default_rng(seed)
    while len(rows) < min(want, n - 1):
        rows.add(int(rng.integers(1, n)))
    return np.array(sorted(rows), np.int32)


def dump_rows(owned, n, budget_bytes=48 << 20, seed=20240):
    """row ids of the output sample, drawn from the rows this rank filled: the same for every build at a given n and
    number of ranks, as many full float64 rows (n columns) as fit the budget"""
    rng = np.random.default_rng(seed)
    return np.sort(rng.choice(owned, size=min(len(owned), max(1, budget_bytes // (8 * n))), replace=False))


def dump_outputs(out_dir, kmat, npos, nneg):
    """what the caller of gkm_main_pywrapper received: rows of its matrix (strict lower triangle, unit diagonal, nothing
    above) at dump_rows, and the (npos, nneg) pair the call wrote into kmat_size.  A sharded call fills only the rows of
    this rank's chunks (their unit diagonal tells which); the sample is drawn from those"""
    os.makedirs(out_dir, exist_ok=True)
    rows = dump_rows(np.flatnonzero(np.diagonal(kmat) == 1.0), kmat.shape[0])
    np.save(os.path.join(out_dir, "kmat_rows.npy"), np.ascontiguousarray(kmat[rows], np.float64))
    np.save(os.path.join(out_dir, "kmat_row_ids.npy"), rows.astype(np.float64))
    np.save(os.path.join(out_dir, "kmat_size.npy"), np.array([npos, nneg], np.float64))


def check_parity(h, kmat, hist_of_rows, n, layout, threads, owned_only=True, want=96):
    """rows of the matrix the product returned (and their integer histograms) against the reference's own numbers"""
    nblk, blk_cols = layout[0], layout[1] or n
    rows = parity_rows(n, blk_cols, nblk, want=want)
    if owned_only:   # a sharded call fills only the rows of this rank's chunks: their unit diagonal tells which
        rows = rows[[kmat[r, r] == 1.0 for r in rows]]
    Kref, Href, t = h.rows_values(rows, threads)
    max_rel, hist_ok, bad = 0.0, True, []
    for i, r in enumerate(rows):
        got, ref = kmat[r, :r], Kref[i, :r]
        if not np.array_equal(got, ref):
            rel = float(np.max(np.abs(got - ref) / np.maximum(np.abs(ref), 1e-300)))
            max_rel = max(max_rel, rel)
            bad.append(int(r))
        if kmat[r, r] != 1.0 or (r + 1 < kmat.shape[1] and kmat[r, r + 1:].any()):
            bad.append(int(r))   # unit diagonal, untouched upper triangle (gkmkern_pylib.c:169-221)
        Hg = hist_of_rows(int(r))            # [r, d+1]
        if not np.array_equal(Hg, Href[i, :, :r].T):
            hist_ok = False
            bad.append(int(r))
    hits = None
    return {"rows": int(len(rows)), "entries": int(rows.sum()), "hist_bit_exact": bool(hist_ok), "kmat_max_rel": max_rel,
            "kmat_bit_identical": max_rel == 0.0 and not bad, "mismatching_rows": sorted(set(bad))[:8],
            "against": "oracle/_ref (unmodified reference): gkmkernel_kernelfunc_batch_all for the doubles, kmertree_dfs mmprofile for the integers",
            "row_set": "rows 1, 2, n-2, n-1; cb-1, cb, cb+1 of every index column block (%d blocks of %d columns); both sides of "
                       "chunk boundaries (multiples of 148 / 592 rows); random rows" % (nblk, blk_cols),
            "reference_seconds": t, "ok": bool(hist_ok and max_rel <= 1e-9 and not bad)}, hits


# ---------------------------------------------------------------------------------------- main
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--n", type=int, default=0, help="override the number of sequences (debugging only)")
    ap.add_argument("--e2e-steps", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-cpu-full", action="store_true", help="skip the full unsampled reference run of configs[1] (~1 min)")
    ap.add_argument("--no-secondary", action="store_true")
    ap.add_argument("--no-parity", action="store_true", help="profiling runs only")
    ap.add_argument("--no-e2e", action="store_true", help="profiling runs only: skip the end-to-end leg")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed gkm_main_pywrapper call returned to DIR/<name>.npy (float64): a fixed, "
                         "seeded sample of rows of the kernel matrix, their row ids and (npos, nneg) -- to compare two builds")
    args = ap.parse_args()
    if args.dump_outputs and args.no_e2e:
        ap.error("--dump-outputs writes what the end-to-end call returned: it cannot be combined with --no-e2e")

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    n = args.n or BASE_N
    total_entries = n * (n - 1) // 2
    config = {"workload": "BASELINE configs[3]: gkm kernel matrix, %d synthetic 300-bp seqs (%d pos + %d neg), strict lower triangle "
                          "(%d x %d), kernel type 2 (EST_TRUNC) L=11 k=7 d=3; the same problem at every N" % (n, n // 2, n - n // 2, n, n),
              "n_seqs": n, "entries_per_step": total_entries, "lmer_pairs_per_entry": PAIRS_PER_ENTRY,
              "sharding": "chunks of row tiles round-robin over %d rank(s), no collective" % world,
              "l2": "L2 flushed (256 MB memset) before every timed pass; %d MB of output written per pass"
                    % (n * n * 8 // (1 << 20)),
              "resident_excludes": "pack + H2D + sqnorm + index build happen once before the timed passes (about 3 % of a pass at 10k; "
                                   "e2e includes them every step)"}

    tmp = tempfile.mkdtemp(prefix="gkmbench_", dir="/dev/shm" if os.path.isdir("/dev/shm") else None)
    pos, neg = write_problem(tmp, n)
    threads = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)

    # ------------------------------------------------------------------ reference arm
    if args.impl == "reference":
        if rank != 0:
            import shutil
            shutil.rmtree(tmp, ignore_errors=True)
            return
        budget = max(2.0, min(30.0, 150.0 / max(1, args.steps + args.warmup)))
        h = open_reference(pos, neg)
        vals, r = [], None
        if h is None:
            r = port_rate(pos, neg, n)
            vals = [r["value"]]
        else:
            try:
                for it in range(args.warmup + args.steps):
                    r = reference_rate(h, n, budget, threads)
                    if it >= args.warmup:
                        vals.append(r["value"])
                r["setup_s"] = h.open_s
                r["setup"] = "read FASTA, per-sequence sqnorm and k-mer tree over all %d sequences: %.1f s, once, not in the rate" % (n, h.open_s)
            finally:
                h.close()
        v = float(np.mean(vals))
        r["value"] = v
        per_step_ms = 1e3 * total_entries / v
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": v, "unit": "entries/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": per_step_ms,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int32+f64", "data": "synthetic",
            "config": config, "cpu_baseline": r,
            "e2e": {"value": v, "unit": "entries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}))
        import shutil
        shutil.rmtree(tmp, ignore_errors=True)
        return

    # ------------------------------------------------------------------ our arm
    from gkmqc_b200 import capi
    lib = capi.load()
    if capi.device_count() < 1:
        raise SystemExit("bench.py: no B200 visible and the product has no CPU fallback: " + capi.last_error())
    ids = (ctypes.c_int * 1)(local_rank)
    if lib.gkmb200_set_devices(ids, 1) != 0:
        raise SystemExit(capi.last_error())
    os.environ["GKM_SHARD"] = "%d/%d" % (rank, world)   # read by gkm_main_pywrapper's problem only
    dist = dist_setup(world)
    verbosity = int(os.environ.get("GKM_BENCH_V", "0"))

    P = capi.Problem(KTYPE, L, K, D)
    P.read(pos, neg)
    P.set_shard(rank, world)
    P.upload()

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)

    # value: resident passes, CUDA events, L2 flushed between passes
    dist_barrier(dist)
    ms = P.bench_lower_resident(args.steps, max(args.warmup, 3), flush_l2=True)
    st = P.stats()
    layout = P.index_layout()
    my_ms = float(ms.sum())
    dist_barrier(dist)
    t_max = dist_max(dist, my_ms)
    launches_per_step = int(dist_sum(dist, st["launches"]))
    value = total_entries * args.steps / (t_max * 1e-3)
    ms_per_step = t_max / args.steps

    # e2e: the drop-in call with host buffers (fresh, untouched output matrix every step, like gkmsvm.py:75)
    e2e_steps = args.e2e_steps or max(1, min(args.steps, 3))
    walls, kmat, e2e_stats = [], None, None
    h2d = d2h = 0
    for it in range(0 if args.no_e2e else 1 + e2e_steps):
        kmat = None
        kmat = np.zeros((n, n))
        dist_barrier(dist)
        t0 = time.perf_counter()
        # nthreads is gkmQC's own default (bin/gkmqc.py:107,162: 1); the library sizes its copy-out threads by the host's cores
        ret, kmat, npos, nneg = capi.main_pywrapper(pos, neg, kernel_type=KTYPE, L=L, k=K, d=D, nthreads=1, verbosity=verbosity, kmat=kmat)
        t1 = time.perf_counter()
        if ret != 0:
            raise SystemExit("gkm_main_pywrapper failed: " + capi.last_error())
        if it > 0:
            walls.append(dist_max(dist, t1 - t0))
        pst = capi.gkmb200_stats()
        lib.gkmb200_get_stats(None, ctypes.byref(pst))
        h2d, d2h = int(pst.h2d_bytes), int(pst.d2h_bytes)
        e2e_stats = pst.as_dict()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, kmat, npos, nneg)
    if args.no_e2e:
        walls = [float("nan")]
    e2e_value = total_entries / float(np.mean(walls))
    h2d = int(dist_sum(dist, h2d))
    d2h = int(dist_sum(dist, d2h))
    clocks = sampler.finish() if rank == 0 else None

    # ---- configs[4], batch scoring (SURVEY.md 8f/f1): every rank scores its own 125k test rows against the same 10k SVs,
    # decision values reduced on the device; at N = 8 that is the 1M x 10k problem
    scoring = None
    if not args.no_secondary and not args.n:
        sv = synth(NSV, seed=99)
        test = synth(NTEST_PER_GPU, seed=1000 + rank)
        alpha = np.random.default_rng(3).standard_normal(NSV)
        with capi.Problem(KTYPE, L, K, D) as PS:
            t0 = time.perf_counter()
            PS.add_block(sv)
            PS.add_block(test)
            t_add = time.perf_counter() - t0
            PS.upload()
            PS.decision_values(NSV, 2368, 0, NSV, alpha, bias=-0.1)   # builds the SV index, sizes the scratch
            dist_barrier(dist)
            t0 = time.perf_counter()
            dv = PS.decision_values(NSV, NTEST_PER_GPU, 0, NSV, alpha, bias=-0.1)
            dt = dist_max(dist, time.perf_counter() - t0)
            scoring = {"workload": "BASELINE configs[4]: %d test x %d SV per GPU (%d test rows in all), fused decision values"
                                   % (NTEST_PER_GPU, NSV, NTEST_PER_GPU * world),
                       "value": NTEST_PER_GPU * world * NSV / dt, "unit": "entries/s", "seconds": dt, "scaling": "weak",
                       "add_sequences_s": t_add, "d2h_bytes": 8 * NTEST_PER_GPU * world}
            if rank == 0 and not args.no_parity:   # sampled test rows against the reference: SVs first, then the rows (SURVEY.md 8c)
                pick = np.unique(np.linspace(0, NTEST_PER_GPU - 1, 48).astype(int))
                p2, n2 = os.path.join(tmp, "sv.fa"), os.path.join(tmp, "tests.fa")
                write_fasta(p2, sv, 0)
                write_fasta(n2, test[pick], NSV)
                hs = open_reference(p2, n2)
                if hs is not None:
                    try:
                        rows = np.arange(NSV, NSV + len(pick), dtype=np.int32)
                        Kr, _, tref = hs.rows_values(rows, threads, endcap=NSV, with_hist=False)
                        want = Kr @ alpha - 0.1
                        rel = float(np.max(np.abs(dv[pick] - want) / np.maximum(np.abs(want), 1e-12)))
                        scoring["parity"] = {"rows": int(len(pick)), "max_rel": rel, "ok": bool(rel <= 1e-9),
                                             "against": "oracle/_ref batch_all(test, 0, nSV) @ alpha + b"}
                        if not args.no_cpu_baseline and world == 1:
                            rb = reference_rate(hs, NSV + len(pick), 6.0, threads, endcap=NSV)
                            scoring["cpu_baseline"] = rb
                    finally:
                        hs.close()

    if dist is not None:   # the last collective is behind us: what follows is rank 0's own reporting
        dist.barrier()
        dist.destroy_process_group()
        dist = None
    if rank != 0:
        import shutil
        shutil.rmtree(tmp, ignore_errors=True)
        return

    # ------------------------------------------------------------------ parity of what the e2e call returned + CPU baseline
    parity, cpu, hits_per_entry = None, None, None
    href = None
    if (not args.no_parity and kmat is not None) or not args.no_cpu_baseline:
        href = open_reference(pos, neg)
    try:
        if not args.no_parity and kmat is not None and href is not None:
            def hist_of_row(r):
                return P.hist_block(r, 1, 0, r)[0]
            P.set_shard(0, 1)
            parity, _ = check_parity(href, kmat, hist_of_row, n, layout, threads, owned_only=world > 1, want=min(96 * world, 800))  # ~96 rows land in rank 0's chunks
            parity["checked"] = "the numpy matrix returned by the timed gkm_main_pywrapper call (rank 0's rows)" + \
                                (" of %d ranks" % world if world > 1 else "")
            # hits per entry of this input, exactly: the histogram of one band of rows, all bins (unit weights: one per L-mer pair within d)
            r0 = min(n - 1, 30000)
            Hb = P.hist_block(r0, min(8, n - r0), 0, r0)
            hits_per_entry = float(Hb.sum()) / float(Hb.shape[0] * Hb.shape[1])
        elif not args.no_parity and kmat is not None:
            parity = {"ok": None, "unavailable": "oracle/_ref was not built on this box"}
        kmat = None
        if world == 1 and not args.no_cpu_baseline:
            if href is not None:
                cpu = reference_rate(href, n, 15.0, threads)
                one = reference_rate(href, n, 5.0, 1)   # SURVEY.md 8d: the 1-thread figure beside the all-cores one
                cpu["single_thread"] = {"value": one["value"], "unit": one["unit"], "kind": one["kind"], "sample": one["sample"]}
                cpu["setup_s"] = href.open_s
            else:
                cpu = port_rate(pos, neg, n)
    finally:
        if href is not None:
            href.close()

    # ------------------------------------------------------------------ roofline of the dominant kernel (DESIGN.md 4)
    variant = VARIANTS.get(st["kernel_variant"], "?")
    peaks = measured_peaks()
    peak_lop3 = capi.microbench("lop3")       # 1e9 lane-ops/s on this GPU, measured now
    peak_popc = capi.microbench("popc")
    per_gpu_entries_s = value / world
    int_alu_equiv = per_gpu_entries_s * PAIRS_PER_ENTRY * INT_OPS_PER_PAIR / 1e9
    ncu, traffic = None, None
    tf = os.path.join(ROOT, "profiles", "ncu_dominant_kernel.json")   # summary of the committed ncu --set full capture
    if os.path.exists(tf):
        try:
            cap = json.load(open(tf))
            if cap.get("variant", "diag") == variant and cap.get("source_sha256") == kernel_source_hash():
                ncu = dict(cap, source="committed capture profiles/ncu_dominant_kernel.json of this kernel source (sha256 %s), not measured in this run" % cap.get("source_sha256"))
                traffic = cap.get("dram_bytes_per_launch")
            else:
                ncu = {"unavailable": "profiles/ncu_dominant_kernel.json was captured on another build of the kernel (variant %s, source %s; this run: %s, %s)"
                                      % (cap.get("variant"), cap.get("source_sha256"), variant, kernel_source_hash())}
        except Exception as e:
            ncu = {"unavailable": str(e)}
    launches_mine = max(1, st["launches"])
    avg_launch_ms = ms_per_step / launches_mine   # two compute streams overlap launches: this is pass time / launches
    if variant == "index":
        peak_gather = capi.microbench("gather16")     # 1e9 random 16-byte gathers (one 32-byte sector each) per second
        probes, sectors = index_probe_counts(L, D, 8)
        nq = SEQLEN - L + 1
        nblk, blk_cols = layout[0], max(1, layout[1])
        # a row probes every column block that starts below it (strict lower triangle)
        probed_blocks = float(sum(min(nblk, (a + blk_cols - 1) // blk_cols) for a in range(1, n))) / world
        sector_bytes = probed_blocks * nq * sectors * 32.0   # algorithmic: distinct sectors the probes of one pass must fetch
        achieved = sector_bytes / (ms_per_step * 1e-3) / 1e9
        hpe = hits_per_entry if hits_per_entry is not None else PAIRS_PER_ENTRY * probes / 4.0 ** L
        hits = hpe * total_entries / world
        # lanes that are on in the shared atomic of a posting: the postings a probe finds in the wanted range, over the slot's four positions
        lanes_on = 32.0 * hits / (probed_blocks * nq * probes) / 4.0
        atoms_kind = "atoms7" if lanes_on < 10.5 else "atoms14"
        peak_atoms = capi.microbench(atoms_kind)      # 1e9 shared-memory atomic adds per second at ~7 / ~14 active lanes of 32, random columns
        sector_frac = achieved / (peak_gather * 32.0)
        hits_rate = hits / (ms_per_step * 1e-3) / 1e9
        hits_frac = hits_rate / peak_atoms
        # Top level = the side of the L1TEX pipe that is closer to its own peak.  `hits` is the algorithmic one (one shared atomic per
        # L-mer pair within d, whatever the layout); the sector traffic depends on how the columns are cut into index blocks
        # (fewer, wider blocks: fewer probes per row), so its fraction FALLS when the layout improves.
        binding = "hits" if hits_frac >= sector_frac else "sectors"
        top = ({"achieved": hits_rate, "peak": peak_atoms, "unit": "G shared atomics/s", "frac": hits_frac} if binding == "hits" else
               {"achieved": achieved, "peak": peak_gather * 32.0, "unit": "GB/s", "frac": sector_frac})
        roofline = {"bound": "l1tex", "binding": binding, "achieved": top["achieved"], "peak": top["peak"], "unit": top["unit"],
                    "frac": top["frac"], "traffic": traffic,
                    "sectors": {"achieved_gbs": achieved, "peak_gbs": peak_gather * 32.0, "frac": sector_frac},
                    "traffic_note": "DRAM bytes per launch from the committed ncu capture (444 rows against one full column block): the output alone is "
                                    "8 B x 444 x 22 528 = 80 MB; the rest is the global scratch of the two cold bins (m <= d - 2: zeroed, then read back by the "
                                    "epilogue, 80 MB that L2 does not always keep) and the 33.5 MB slot table fetched once per launch -- ~90 GB/s in all, "
                                    "1.4 %% of HBM bandwidth (MEASURED_PEAKS hbm_gbs = %s): not what bounds this kernel" % peaks.get("hbm_gbs"),
                    "note": "index variant: every forward L-mer of a row probes %d 8-byte slots (%d distinct 32-byte sectors) of every L2-resident "
                            "column-block table that starts below the row; sectors.achieved = sum over rows of blocks x %d L-mers x sectors x 32 B per pass / time; "
                            "sectors.peak = random 16-byte gathers from a 64 MB table measured in this run (x 32 B per sector): a UTILISATION of the L1TEX "
                            "gather ceiling by implementation traffic, not algorithmic work. The irreducible part is `hits` (one shared atomic per "
                            "L-mer pair within d). Slot loads and shared atomics are wavefronts of the same L1TEX data pipe: the two fractions add up "
                            "to the pipe's load, neither reaches 1 alone; achieved / peak / frac at the top are those of `binding`, the larger one" % (probes, sectors, nq),
                    "probes_per_lmer": probes, "sectors_per_lmer": sectors, "peak_gather_gsectors": peak_gather,
                    "index_blocks": nblk, "index_block_cols": blk_cols,
                    "hits": {"per_entry": hpe, "per_entry_source": "gkmb200_hist_block on 8 rows of this input" if hits_per_entry is not None else "uniform-sequence expectation",
                             "per_pass": hits, "lanes_on_per_atomic": lanes_on, "achieved_ghits_s": hits_rate, "peak_gatoms_s": peak_atoms,
                             "frac": hits_frac,
                             "note": "peak = shared-memory atomic adds with ~%d of 32 lanes on per warp instruction, random columns of an 80 KB histogram row, two CTAs "
                                     "of 1024 threads per SM (gkmb200_microbench %s): the pattern of the hot loop at this problem size"
                                     % (7 if atoms_kind == "atoms7" else 14, atoms_kind)},
                    "int_alu_equivalent": {"achieved_gops": int_alu_equiv, "peak_lop3_gops": peak_lop3, "ratio": int_alu_equiv / peak_lop3,
                                           "note": "SURVEY.md 8d's unit, labelled as such: what the canonical 5-op XOR/POPC form would need for the same "
                                                   "entries/s; the index variant never touches pairs farther apart than d, so this is not a utilisation"},
                    "hbm": {"algorithmic_bytes_per_entry": 8, "achieved_gbs": per_gpu_entries_s * 8 / 1e9, "peak_gbs": peaks.get("hbm_gbs"),
                            "frac": (per_gpu_entries_s * 8 / 1e9 / peaks["hbm_gbs"]) if peaks.get("hbm_gbs") else None},
                    "ncu": ncu, "avg_launch_ms": avg_launch_ms, "kernel_variant": variant}
    else:
        roofline = {"bound": "int_alu", "achieved": int_alu_equiv, "peak": peak_lop3, "unit": "Gop/s", "frac": int_alu_equiv / peak_lop3,
                    "traffic": traffic,
                    "note": "achieved = entries/s x 168200 L-mer pairs x 5 integer ops of the canonical XOR/LOP3/POPC form "
                            "(SURVEY.md 8d); peak = LOP3 lane-ops/s measured in this run (MEASURED_PEAKS.json has no integer "
                            "peak). The bit-sliced kernel needs < 1 op per pair, so frac > 1 is possible; see DESIGN.md",
                    "peak_popc_gops": peak_popc, "ncu": ncu, "avg_launch_ms": avg_launch_ms, "kernel_variant": variant}

    # ------------------------------------------------------------------ secondary figures (rank 0, N = 1 only)
    secondary = None
    if world == 1 and not args.no_secondary and not args.n:
        secondary = {}
        n2 = SECOND_N
        e2 = n2 * (n2 - 1) // 2
        pos2, neg2 = write_problem(tmp, n2, tag="_10k")

        def e2e_of(posf, negf, nn, reps=3, **kw):
            w = []
            for it in range(reps + 1):
                km = np.zeros((nn, nn))
                t0 = time.perf_counter()
                ret, km, _, _ = capi.main_pywrapper(posf, negf, nthreads=1, verbosity=verbosity, kmat=km, **kw)
                if ret != 0:
                    raise SystemExit("gkm_main_pywrapper failed: " + capi.last_error())
                if it > 0:
                    w.append(time.perf_counter() - t0)
                del km
            return float(np.mean(w))

        # configs[1]: 5k + 5k x 300 bp, the workload round 1 reported
        with capi.Problem(KTYPE, L, K, D) as P2:
            P2.read(pos2, neg2)
            m2 = P2.bench_lower_resident(3, 2, flush_l2=True)
        w2 = e2e_of(pos2, neg2, n2, kernel_type=KTYPE, L=L, k=K, d=D)
        sec1 = {"workload": "BASELINE configs[1]: 5k + 5k x 300 bp, type 2, L=11 k=7 d=3", "value": e2 / (float(m2.mean()) * 1e-3),
                "ms_per_step": float(m2.mean()), "e2e": {"value": e2 / w2, "ms_per_step": 1e3 * w2}, "unit": "entries/s"}
        # a caller pinned to ONE core (a slurm job that asked for one): the copy-out runs on that core alone
        try:
            full_mask = os.sched_getaffinity(0)
            os.sched_setaffinity(0, {sorted(full_mask)[0]})
            try:
                w1 = e2e_of(pos2, neg2, n2, reps=2, kernel_type=KTYPE, L=L, k=K, d=D)
            finally:
                os.sched_setaffinity(0, full_mask)
            sec1["e2e_one_core"] = {"value": e2 / w1, "ms_per_step": 1e3 * w1, "note": "same call with the process's affinity mask cut to one core"}
        except Exception as e:
            sec1["e2e_one_core"] = {"error": str(e)}
        with capi.Problem(4, L, K, D, 50, 50.0, 1.0) as P4:
            P4.read(pos2, neg2)
            ms4 = P4.bench_lower_resident(3, 2, flush_l2=True)
            sec1["type4"] = {"value": e2 / (float(ms4.mean()) * 1e-3), "ms_per_step": float(ms4.mean()),
                             "note": "wgkm (EST_TRUNC_PW, M=50 H=50) on the same sequences, resident pass"}
        if not args.no_cpu_baseline and not args.no_cpu_full:
            try:   # SURVEY.md 8d: the unmodified reference through the same ctypes call on the same files, all rows, nothing sampled
                import pyoracle
                if pyoracle.have_ref():
                    kmr = np.zeros((n2, n2))
                    t0 = time.perf_counter()
                    ret, kmr, _, _ = pyoracle.call_pywrapper(pyoracle.ref_pywrapper(), pos2, neg2, kernel_type=KTYPE, L=L, k=K, d=D,
                                                             nthreads=threads, verbosity=0, kmat=kmr)
                    tr = time.perf_counter() - t0
                    kmo = np.zeros((n2, n2))
                    ret2, kmo, _, _ = capi.main_pywrapper(pos2, neg2, kernel_type=KTYPE, L=L, k=K, d=D, nthreads=1, verbosity=0, kmat=kmo)
                    sec1["cpu_full"] = {"value": e2 / tr, "unit": "entries/s", "seconds": tr, "cores": threads, "kind": "reference",
                                        "call": "oracle/_ref/gkmkern_pylib.so::gkm_main_pywrapper on the same FASTA files, every row, nthreads = all cores",
                                        "whole_matrix_identical_to_ours": bool(ret == 0 and ret2 == 0 and np.array_equal(kmr, kmo)),
                                        "e2e_ratio": tr / w2}
                    del kmr, kmo
            except Exception as e:
                sec1["cpu_full"] = {"error": str(e)}
        secondary["configs1_10k"] = sec1

        # gkmQC's real default (bin/gkmqc.py:154,169-199): wgkm type 4, L=10 k=6 d=3, 600-bp window, 5k + 5k
        posd, negd = write_problem(tmp, n2, seed=4321, seqlen=600, tag="_600")
        with capi.Problem(4, 10, 6, 3, 50, 50.0, 1.0) as Pd:
            Pd.read(posd, negd)
            md = Pd.bench_lower_resident(3, 2, flush_l2=True)
            vd = VARIANTS.get(Pd.stats()["kernel_variant"], "?")
        wd = e2e_of(posd, negd, n2, kernel_type=4, L=10, k=6, d=3, M=50, H=50.0)
        pairs600 = (600 - 10 + 1) * 2 * (600 - 10 + 1)
        secondary["gkmqc_default"] = {"workload": "gkmQC default: wgkm (type 4, M=50 H=50) L=10 k=6 d=3, 5k + 5k x 600 bp", "unit": "entries/s",
                                      "value": e2 / (float(md.mean()) * 1e-3), "ms_per_step": float(md.mean()), "kernel_variant": vd,
                                      "e2e": {"value": e2 / wd, "ms_per_step": 1e3 * wd},
                                      "lmer_pairs_per_entry": pairs600, "lmer_pairs_per_s": e2 / (float(md.mean()) * 1e-3) * pairs600,
                                      "type4_300bp_L11_lmer_pairs_per_s": sec1["type4"]["value"] * PAIRS_PER_ENTRY}

        # the consumer of the matrix (SURVEY.md 8f/f4): gkmQC's 5-fold x 10-repeat C-SVC cross-validation on the matrix kept
        # resident on the device, gkmQC's default kernel; two of the 50 fits against sklearn's SVC on the same splits
        try:
            from sklearn.metrics import roc_auc_score
            from sklearn.model_selection import StratifiedKFold
            from sklearn.svm import SVC
            rng = np.random.default_rng(7)
            arrm = synth(n2)
            npos_m = n2 // 2
            motifs = [b"GATAAGGCAT", b"TTGACGTCAA", b"CCCGCCCCTA"]
            for i in range(npos_m):   # degenerate motifs planted in the positives: a problem an SVM can learn
                for m in motifs[: 1 + i % 3]:
                    at = int(rng.integers(0, 290))
                    mm = bytearray(m)
                    if rng.random() < 0.5:
                        mm[int(rng.integers(0, 10))] = b"ACGT"[int(rng.integers(0, 4))]
                    arrm[i, at:at + 10] = np.frombuffer(bytes(mm), np.uint8)
            ym = np.concatenate((np.ones(npos_m, int), np.zeros(n2 - npos_m, int)))
            splits = []
            for rep in range(10):
                splits.extend(StratifiedKFold(n_splits=5, shuffle=True, random_state=rep).split(np.zeros(n2), ym))
            with capi.Problem(4, 10, 6, 3, 50, 50.0, 1.0) as Pm:
                Pm.add_block(arrm)
                Pm.upload()
                t0 = time.perf_counter()
                scores, fits, _ = capi.svm_cv(ym, splits, problem=Pm, C=1.0, eps=1e-3)
                t_first = time.perf_counter() - t0
                t0 = time.perf_counter()
                scores, fits, _ = capi.svm_cv(ym, splits, problem=Pm, C=1.0, eps=1e-3)
                t_fits = time.perf_counter() - t0
                aucs = [roc_auc_score(ym[te], sc) for (_, te), sc in zip(splits, scores)]
                Km = Pm.kernel_lower()
                Km = np.maximum(Km, Km.T)
            t0 = time.perf_counter()
            worst = 0.0
            for f_i, (tr, te) in enumerate(splits[:2]):
                sv = SVC(kernel="precomputed", C=1.0, tol=1e-3, shrinking=False, gamma=1.0, cache_size=1000)
                ref_s = sv.fit(Km[tr][:, tr], ym[tr]).decision_function(Km[te][:, tr])
                worst = max(worst, float(np.max(np.abs(ref_s - scores[f_i]))))
            t_sk = time.perf_counter() - t0
            del Km
            secondary["svm_cv"] = {"workload": "50 C-SVC fits (5-fold x 10 repeats, C = 1, tol = 1e-3) on 10k x 300 bp with planted motifs, wgkm L=10 k=6 d=3, matrix resident on the device",
                                   "fits_s": t_fits, "with_matrix_s": t_first, "auc_mean": float(np.mean(aucs)),
                                   "iterations_mean": float(np.mean([f["n_iter"] for f in fits])), "n_sv_mean": float(np.mean([f["n_sv"] for f in fits])),
                                   "sklearn_2_fits_s": t_sk, "max_abs_diff_decision_values_vs_sklearn": worst}
        except Exception as e:
            secondary["svm_cv"] = {"error": str(e)}

        # genome-like, NON-uniform input (AT-rich background, a repeat family in 20 %, poly-A tracts in 10 %, dinucleotide repeats in 5 %, 5 % duplicates)
        try:
            import importlib.util
            spec = importlib.util.spec_from_file_location("nonuniform", os.path.join(ROOT, "tools", "nonuniform.py"))
            nu = importlib.util.module_from_spec(spec)
            spec.loader.exec_module(nu)
            x = nu.workloads(n2)["mixed"]
            with capi.Problem(KTYPE, L, K, D) as Pn:
                Pn.add_block(nu.ACGT[x])
                msn = Pn.bench_lower_resident(2, 1, flush_l2=True)
                secondary["nonuniform"] = {"workload": "10k x 300 bp, mixed (tools/nonuniform.py)", "value": e2 / (float(msn.mean()) * 1e-3), "unit": "entries/s",
                                           "ms_per_step": float(msn.mean()), "kernel_variant": VARIANTS.get(Pn.stats()["kernel_variant"], "?"),
                                           "note": "resident pass, kernel type 2; bit-exact against the bit-sliced kernel in tests/test_gpu_parity.py::test_nonuniform_index_vs_bitsliced"}
        except Exception as e:   # a reporting extra must not take the bench line down
            secondary["nonuniform"] = {"error": str(e)}
    P.close()

    out = {
        "metric": METRIC, "value": value, "unit": "entries/s",
        "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms_per_step,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int32+f64", "data": "synthetic",
        "config": config, "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": "entries/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": 1e3 * float(np.mean(walls)), "steps": e2e_steps,
                "call": "gkm_main_pywrapper(FASTA paths, double** rows of a fresh numpy matrix, int[2])",
                "host": {"cores": threads, "thp": thp_mode(),
                         "copy_threads": e2e_stats and e2e_stats["copy_threads"], "thp_chunks": e2e_stats and e2e_stats["thp_chunks"],
                         "scatter_ms": e2e_stats and e2e_stats["scatter_ms"], "gpu_wait_ms": e2e_stats and e2e_stats["wait_ms"],
                         "kernel_ms": e2e_stats and e2e_stats["kernel_ms"],
                         "first_touch_gbs": (e2e_stats["d2h_bytes"] / 1e6 / e2e_stats["scatter_ms"]) if e2e_stats and e2e_stats["scatter_ms"] else None,
                         "note": "rank 0's last call: the copy-out writes a fresh np.zeros matrix, i.e. page faults (tools/pagefault_probe.c)"}},
        "gpu_launches": launches_per_step * args.steps, "parity": parity, "roofline": roofline, "cpu_baseline": cpu,
        "scoring": scoring, "secondary": secondary}
    print(json.dumps(out))
    sys.stdout.flush()
    try:
        import shutil
        shutil.rmtree(tmp, ignore_errors=True)
    except Exception:
        pass
    if parity is not None and parity.get("ok") is False:
        sys.stderr.write("bench.py: PARITY FAILURE against the reference: %s\n" % json.dumps(parity))
        raise SystemExit(3)
    if scoring and scoring.get("parity") and scoring["parity"]["ok"] is False:
        sys.stderr.write("bench.py: PARITY FAILURE (scoring) against the reference: %s\n" % json.dumps(scoring["parity"]))
        raise SystemExit(3)


if __name__ == "__main__":
    main()
