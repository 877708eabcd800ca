"""Host-side mirror of the reference's caller of the path (scripts/gkmsvm.py:67-99, ``computeGkmKernel``).

Same function name, same positional argument list and same return triple as the reference's driver, so the
parity tests read like its own code path, but bound to gkmqc_b200/bin/gkmkern_pylib.so.  The reference's
module itself works unchanged against this library (INTEGRATION.md section 1); this mirror exists because the
GPU box has no copy of the reference tree.  ``crossValidate`` mirrors the consumer of the matrix
(gkmsvm.py:104-176) with the GPU solver of SURVEY.md 8f/f4 in place of the multiprocessing pool of sklearn SVCs.
"""
import logging
import sys

import numpy as np

from . import capi

MAX_SEQS = 15000  # the reference allocates a fixed 15000 x 15000 matrix per call (gkmsvm.py:75)


def computeGkmKernel(args_gkm, max_seqs=MAX_SEQS):
    """args_gkm = [kernel_type, L, k, d, M, H, gamma, posfile, negfile, nthreads, verbosity]
    (the list gkmsvm.init builds, gkmsvm.py:183-195).  Returns (kmat, n_pseqs, n_nseqs): the symmetric
    n x n kernel matrix with unit diagonal, cut out of the padded matrix the C side filled."""
    kernel_type, L, k, d, M, H, gamma, posfile, negfile, nthreads, verbosity = args_gkm
    ret, padded, n_pseqs, n_nseqs = capi.main_pywrapper(
        posfile, negfile, kernel_type=kernel_type, L=L, k=k, d=d, M=M, H=H, gamma=gamma,
        nthreads=nthreads, verbosity=verbosity, nmax=max_seqs)
    if ret:
        logging.error("error on kernel construction")  # gkmsvm.py:90-92
        sys.exit()
    n = n_pseqs + n_nseqs
    kmat = padded[:n, :n]
    return np.maximum(kmat, kmat.T), n_pseqs, n_nseqs  # lower triangle -> symmetric (gkmsvm.py:96-97)


def crossValidate(args_svm, _kmat, n_pseqs, n_nseqs, problem=None):
    """args_svm = [regularization, precision, shrinking, cache_size, ncv, repeats, fast_estimation, random_seeds, p]
    (gkmsvm.py:198-208).  Same splits as the reference (StratifiedKFold per repeat, gkmsvm.py:146-150), same
    (mean AUC, std AUC) result; the 5 x 10 C-SVC fits run concurrently on the GPU through gkmb200_svm_cv_ex.
    _kmat = the symmetric host matrix, or None with `problem` given: the matrix then never leaves the device.
    shrinking != 0 runs libsvm's shrinking heuristic, as the reference's SVC(shrinking=...) does."""
    from sklearn.metrics import roc_auc_score
    from sklearn.model_selection import StratifiedKFold
    regularization, precision, shrinking, _cache_size, ncv, repeats, fast_estimation, random_seeds, _p = args_svm
    if random_seeds < 0:
        random_seeds = None
    seqids = ["p%4d" % x for x in range(n_pseqs)] + ["n%4d" % x for x in range(n_nseqs)]
    y = np.concatenate((np.repeat(1, n_pseqs), np.repeat(0, n_nseqs)))
    if fast_estimation != 0:
        raise NotImplementedError("fast_estimation is commented out in the reference as well (gkmsvm.py:160-174)")
    splits = []
    for _ in range(repeats):
        kf = StratifiedKFold(n_splits=ncv, shuffle=True, random_state=random_seeds)
        splits.extend(kf.split(seqids, y))
    scores, fits, _ = capi.svm_cv(y, splits, kmat=_kmat, problem=problem, C=regularization, eps=precision,
                                  shrinking=int(bool(shrinking)))
    aucs = []
    for (_, test), s, f in zip(splits, scores, fits):
        aucs.append(roc_auc_score(y[test], s))
        logging.info("SVC training and validation; nu = %.3f, AUC = %.3f", f["nu"], aucs[-1])
    logging.info("done cross-validation.")
    return np.mean(aucs), np.std(aucs)


def init(pos_fa, neg_fa, args, resident=False):
    """gkmsvm.init (gkmsvm.py:182-222): one bin of gkmQC's `evaluate` -- kernel matrix, cross-validation, one line appended to
    `<args.name>.gkmqc.eval.out` (pos_fa, neg_fa, n_pseqs, mean AUC, std AUC; tab-separated).  `args` carries the attributes the
    reference's argparse namespace has (gkmsvm.py:236-300, bin/gkmqc.py:150-215).
    resident=True keeps the matrix on the device between the two steps (gkmb200_svm_cv with kmat = NULL): same numbers, no
    15000 x 15000 host matrix."""
    args_gkm = [args.kernel_type, args.full_word_length, args.non_gap_length, args.max_num_gaps, args.init_decay,
                args.half_life_decay, args.rbf_gamma, pos_fa, neg_fa, args.n_processes, args.verbosity]
    args_svm = [args.regularization, args.precision, args.shrinking, args.cache_size, args.ncv, args.repeats,
                args.fast_estimation, args.random_seeds, args.n_processes]
    logging.info("%s: building up kernel matrix", pos_fa)
    if resident:
        with capi.Problem(args.kernel_type, args.full_word_length, args.non_gap_length, args.max_num_gaps,
                          args.init_decay, args.half_life_decay, args.rbf_gamma) as P:
            n_pseqs = P.read(pos_fa, neg_fa)
            n_nseqs = P.n - n_pseqs
            logging.info("%s: svm training", pos_fa)
            auc_score, auc_std = crossValidate(args_svm, None, n_pseqs, n_nseqs, problem=P)
    else:
        kmat, n_pseqs, n_nseqs = computeGkmKernel(args_gkm)
        logging.info("%s: svm training", pos_fa)
        auc_score, auc_std = crossValidate(args_svm, kmat, n_pseqs, n_nseqs)
    logging.info("%s: writing result to output file", pos_fa)
    with open(args.name + ".gkmqc.eval.out", "a") as fa:
        fa.write("\t".join(map(str, [pos_fa, neg_fa, n_pseqs, auc_score, auc_std])) + "\n")
    return auc_score, auc_std


def main(argv=None):
    """`python -m gkmqc_b200.driver -p pos.fa -n neg.fa -w name ...`: the command line of scripts/gkmsvm.py (gkmsvm.py:224-324:
    same options, same defaults, same output file) on the engine.  --resident (not in the reference) keeps the matrix on the
    device between the kernel and the cross-validation."""
    import argparse
    ap = argparse.ArgumentParser(description="gkm-SVM evaluation of one bin on B200 (option set of gkmQC's scripts/gkmsvm.py)",
                                 formatter_class=argparse.RawTextHelpFormatter)
    ap.add_argument("-p", "--pos-fa", type=str, required=True, help="positive fa file. REQUIRED")
    ap.add_argument("-n", "--neg-fa", type=str, required=True, help="negative fa file. REQUIRED")
    ap.add_argument("-w", "--name", type=str, required=True, help="prefix of output file to write AUC score. REQUIRED")
    ap.add_argument("-s", "--random-seeds", type=int, default=-1, help="random seed number (default: no seed)")
    ap.add_argument("-@", "--n-processes", type=int, default=1, help="number of processes (default: 1)")
    ap.add_argument("-v", "--verbosity", type=int, default=1, help="verbosity (default: 1), 0: silent")
    g = ap.add_argument_group("gkm-kernel")
    g.add_argument("-t", "--kernel-type", type=int, default=4, help="0 gkm, 1 full filter, 2 truncated filter, 3 gkmrbf, 4 wgkm (default), 5 wgkmrbf")
    g.add_argument("-L", "--full-word-length", type=int, default=10, help="full word length including gaps (default: 10)")
    g.add_argument("-k", "--non-gap-length", type=int, default=6, help="number of non-gap positions (default: 6)")
    g.add_argument("-d", "--max-num-gaps", type=int, default=3, help="maximum number of gaps allowed (default: 3)")
    g.add_argument("-M", "--init-decay", type=int, default=50, help="initial value M of the decay function, -t 4 or 5 (default: 50)")
    g.add_argument("-H", "--half-life-decay", type=int, default=50, help="half-life H of the decay function, -t 4 or 5 (default: 50)")
    g.add_argument("-G", "--rbf-gamma", type=float, default=1.0, help="gamma for RBF kernel, -t 3 or 5 (default: 1.0)")
    s = ap.add_argument_group("SVM training")
    s.add_argument("-C", "--regularization", type=float, default=1.0, help="regularization parameter C (default: 1.0)")
    s.add_argument("-e", "--precision", type=float, default=0.001, help="precision parameter epsilon (default: 0.001)")
    s.add_argument("-u", "--shrinking", type=int, default=0, help="use the shrinking heuristic of libsvm, 0 or 1 (default: 0)")
    s.add_argument("-c", "--cache-size", type=int, default=512, help="accepted for compatibility (the matrix is resident)")
    s.add_argument("-x", "--ncv", type=int, default=5, help="x-fold cross validation (default: 5)")
    s.add_argument("-r", "--repeats", type=int, default=1, help="number of repeats of CV training (default: 1)")
    s.add_argument("-f", "--fast-estimation", type=int, default=0, help="not available (commented out in the reference as well)")
    ap.add_argument("--resident", action="store_true", help="keep the kernel matrix on the device (no host matrix)")
    args = ap.parse_args(argv)
    return init(args.pos_fa, args.neg_fa, args, resident=args.resident)


if __name__ == "__main__":
    logging.basicConfig(stream=sys.stdout, format="%(levelname)s %(asctime)s: %(message)s", datefmt="%Y-%m-%d %H:%M:%S",
                        level=logging.INFO)  # formatting compatible with clog (gkmsvm.py:326-333)
    main()
