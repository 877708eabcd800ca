"""libsvm's Solver::Solve with shrinking = 1 (sklearn's SVC(shrinking=True), C-SVC), restated in plain numpy in the
data-parallel form gkm_svm.cu's shrinking solver uses (TEST INFRASTRUCTURE ONLY; no product code):

* every per-iteration loop is a vector operation over the active set [0, active_size), and the arg-max picks keep
  libsvm's tie rule (the last index wins);
* do_shrinking's sequential two-pointer partition is the prefix-count pairing ``shrink_pairs``: the k-th shrunk position
  below n_keep (counted upward) trades places with the k-th kept position at or above n_keep (counted downward);
* reconstruct_gradient keeps libsvm's two loop orders, each inactive G entry summing its terms in libsvm's order (the
  vector runs across the independent entries, never within one sum);
* Q is libsvm's float kernel-row cache: float32(y_i y_k K_ik), promoted to double.

Conventions are those of oracle/pysvm.py: the training ids of a fit in grouped order (label 0 first) with y = +1 for
that class.  ``solve`` returns alpha in that order, rho, the objective, the iteration count and the shrinking statistics
gkmb200_svm_cv_ex reports.
"""
import numpy as np

TAU = 1e-12


def be_shrunk(G, A, y, C, gmax1, gmax2):
    """libsvm's be_shrunk for every element of the given arrays"""
    upper = A >= C
    lower = A <= 0.0
    pos = y > 0
    return np.where(upper, np.where(pos, -G > gmax1, -G > gmax2),
                    np.where(lower, np.where(pos, G > gmax2, G > gmax1), False))


def shrink_pairs(flags):
    """(n_keep, low, high): do_shrinking's partition of an active set whose elements carry the be_shrunk `flags`, as
    pairs of positions to swap -- the k-th shrunk position in [0, n_keep) counted upward with the k-th kept position in
    [n_keep, active_size) counted downward, from one exclusive prefix count of the kept elements"""
    flags = np.asarray(flags, bool)
    keep = ~flags
    n_keep = int(np.count_nonzero(keep))
    P = np.cumsum(keep) - keep                      # kept elements before each position
    pos = np.arange(len(flags))
    m = n_keep - int(P[n_keep]) if n_keep < len(flags) else 0   # shrunk below n_keep = kept at or above it
    low = np.empty(m, np.int64)
    high = np.empty(m, np.int64)
    lo = np.flatnonzero(flags[:n_keep])
    low[pos[lo] - P[lo]] = lo                       # upward rank: shrunk elements before p
    hi = n_keep + np.flatnonzero(keep[n_keep:])
    high[m - 1 - (P[hi] - (n_keep - m))] = hi       # downward rank: kept elements after q
    return n_keep, low, high


def shrink_sequential(flags):
    """libsvm's own loop (do_shrinking after the max reduction) on a vector of be_shrunk flags: (active_size, the
    permutation it leaves) -- the reference shrink_pairs is checked against"""
    f = list(map(bool, flags))
    perm = list(range(len(f)))
    active_size = len(f)
    i = 0
    while i < active_size:
        if f[i]:
            active_size -= 1
            while active_size > i:
                if not f[active_size]:
                    f[i], f[active_size] = f[active_size], f[i]
                    perm[i], perm[active_size] = perm[active_size], perm[i]
                    break
                active_size -= 1
        i += 1
    return active_size, perm


def solve(K, order, y_pm, C, eps, max_iter=-1):
    """one C-SVC fit with shrinking on the training ids `order` (grouped) with labels `y_pm`; returns a dict with alpha
    (grouped order), rho, obj, n_iter and the statistics shrink_passes, min_active, unshrink_iter, recon_a, recon_b"""
    idx = np.array(order, np.int64)
    y = np.array(y_pm, np.int64)
    l = len(idx)
    qd = K[idx, idx].astype(np.float64)             # QD: double, permuted with the rest
    G = np.full(l, -1.0)
    A = np.zeros(l)
    G_bar = np.zeros(l)
    aset = np.arange(l)
    st = dict(shrink_passes=0, min_active=l, unshrink_iter=-1, recon_a=0, recon_b=0)
    state = dict(act=l, unshrink=False)

    def q_row(i, cols):
        return ((y[i] * y[cols]).astype(np.float64) * K[idx[i], idx[cols]]).astype(np.float32).astype(np.float64)

    def reconstruct():
        act = state["act"]
        if act == l:
            return
        G[act:] = G_bar[act:] + -1.0
        free = np.flatnonzero((A[:act] > 0.0) & (A[:act] < C))
        nr_free = len(free)
        inact = np.arange(act, l)
        # libsvm's int arithmetic; below 46 341 points neither side can overflow
        if nr_free * l > 2 * act * (l - act):
            st["recon_a"] += 1
            for j in free:      # order A: row of each inactive i, its free j ascending
                q = ((y[inact] * y[j]).astype(np.float64) * K[idx[inact], idx[j]]).astype(np.float32).astype(np.float64)
                G[act:] = G[act:] + A[j] * q
        else:
            st["recon_b"] += 1
            for i in free:      # order B: row of each free active i ascending, into every inactive j
                G[act:] = G[act:] + A[i] * q_row(i, inact)

    def swap(p, q):
        for arr in (G, A, y, idx, G_bar, aset, qd):
            arr[p], arr[q] = arr[q].copy(), arr[p].copy()

    def do_shrinking(it):
        act = state["act"]
        a, g, yy = A[:act], G[:act], y[:act]
        pos = yy > 0
        up = np.where(pos, a < C, a > 0.0)          # not upper (y = +1) / not lower (y = -1): the -yG of I_up
        low = np.where(pos, a > 0.0, a < C)
        gm1 = np.max(np.where(up, -yy * g, -np.inf), initial=-np.inf)
        gm2 = np.max(np.where(low, yy * g, -np.inf), initial=-np.inf)
        if not state["unshrink"] and gm1 + gm2 <= eps * 10:
            state["unshrink"] = True
            st["unshrink_iter"] = it
            reconstruct()
            state["act"] = act = l
        flags = be_shrunk(G[:act], A[:act], y[:act], C, gm1, gm2)
        n_keep, lo, hi = shrink_pairs(flags)
        for p, q in zip(lo, hi):
            swap(p, q)
        state["act"] = n_keep
        st["shrink_passes"] += 1
        st["min_active"] = min(st["min_active"], n_keep)

    def select():
        act = state["act"]
        a, g, yy = A[:act], G[:act], y[:act]
        pos = yy > 0
        up = np.where(pos, a < C, a > 0.0)
        v = np.where(up, np.where(pos, -g, g), -np.inf)
        gmax = np.max(v, initial=-np.inf)
        if gmax == -np.inf:
            return None
        i = int(np.flatnonzero(v == gmax)[-1])
        qi = q_row(i, np.arange(act))
        low = np.where(pos, a > 0.0, a < C)
        mg = np.where(pos, g, -g)
        gmax2 = np.max(np.where(low, mg, -np.inf))
        gd = np.where(pos, gmax + g, gmax - g)
        qc = np.where(pos, (qd[i] + qd[:act]) - 2.0 * y[i] * qi, (qd[i] + qd[:act]) + 2.0 * y[i] * qi)
        od = np.where(qc > 0.0, (gd * gd) / np.where(qc > 0.0, qc, 1.0), (gd * gd) / TAU)
        cand = low & (gd > 0.0)
        if gmax + gmax2 < eps or not cand.any():
            return None
        w = np.where(cand, od, -np.inf)
        j = int(np.flatnonzero(w == np.max(w))[-1])
        return i, j

    if max_iter < 0:
        max_iter = np.iinfo(np.int64).max
    it = 0
    counter = min(l, 1000) + 1
    while True:
        if it >= max_iter:
            break
        counter -= 1
        if counter == 0:
            counter = min(l, 1000)
            do_shrinking(it)
        ij = select()
        if ij is None:
            reconstruct()
            state["act"] = l
            ij = select()
            if ij is None:
                break
            counter = 1
        it += 1
        i, j = ij
        act = state["act"]
        qi = q_row(i, np.arange(l))
        qj = q_row(j, np.arange(l))
        oai, oaj = A[i], A[j]
        ai, aj = oai, oaj
        if y[i] != y[j]:
            qc = qd[i] + qd[j] + 2.0 * qi[j]
            if qc <= 0:
                qc = TAU
            delta = (-G[i] - G[j]) / qc
            diff = ai - aj
            ai += delta
            aj += delta
            if diff > 0:
                if aj < 0:
                    aj, ai = 0.0, diff
            elif ai < 0:
                ai, aj = 0.0, -diff
            if diff > 0:
                if ai > C:
                    ai, aj = C, C - diff
            elif aj > C:
                aj, ai = C, C + diff
        else:
            qc = qd[i] + qd[j] - 2.0 * qi[j]
            if qc <= 0:
                qc = TAU
            delta = (G[i] - G[j]) / qc
            s = ai + aj
            ai -= delta
            aj += delta
            if s > C:
                if ai > C:
                    ai, aj = C, s - C
            elif aj < 0:
                aj, ai = 0.0, s
            if s > C:
                if aj > C:
                    aj, ai = C, s - C
            elif ai < 0:
                ai, aj = 0.0, s
        A[i], A[j] = ai, aj
        dai, daj = ai - oai, aj - oaj
        G[:act] = G[:act] + (qi[:act] * dai + qj[:act] * daj)
        if (oai >= C) != (ai >= C):
            G_bar[:] = G_bar - C * qi if oai >= C else G_bar + C * qi
        if (oaj >= C) != (aj >= C):
            G_bar[:] = G_bar - C * qj if oaj >= C else G_bar + C * qj

    act = state["act"]
    yG = y[:act] * G[:act]
    a = A[:act]
    free = (a > 0.0) & (a < C)
    if free.any():
        s = 0.0
        for v in yG[free]:      # libsvm's sequential sum
            s += v
        rho = s / np.count_nonzero(free)
    else:
        ub_set = ((a >= C) & (y[:act] < 0)) | ((a <= 0.0) & (y[:act] > 0))
        lb_set = ((a >= C) & (y[:act] > 0)) | ((a <= 0.0) & (y[:act] < 0))
        ub = np.min(yG[ub_set]) if ub_set.any() else np.inf
        lb = np.max(yG[lb_set]) if lb_set.any() else -np.inf
        rho = (ub + lb) / 2
    obj = 0.0
    for k in range(l):
        obj += A[k] * (G[k] + -1.0)
    alpha = np.empty(l)
    alpha[aset] = A
    return dict(alpha=alpha, rho=rho, obj=obj / 2, n_iter=it, **st)
