"""numpy restatement of the L-mer table (gkmqc_b200/csrc/gkm_lmer_table.h) in the header's operation order, so that it
equals the sm_100a kernels and the CPU emulator bit for bit.  Its inputs come from host functions the library exports:
the base codes of a problem's sequences (gkmb200_problem_codes), the positional weights (gkmb200_posweights) and the
mismatch weights w[0..d] (gkmb200_problem_get_weights).

    S[v] = sum_c beta_c sum_{y L-mer of either strand of c, code(y) = v} wt_c(y),  beta_c = alpha_c / |c|
    A_m[u] = sum_{v : ham(u, v) = m} S[v],  T[u] = sum_m w[m] A_m[u]
    score(r) = bias + (sum_{x forward L-mer of r} wt_r(x) T[code(x)]) / |r|
"""
import numpy as np

from gkmqc_b200 import capi


def base_bit(t, L, hi):
    """gkm_idx_base_bit: the code bit that holds bit `hi` of base t of the window"""
    lb = min(L, 2)
    return 2 * t + hi if t < lb else (L if hi else lb) + t


def window_codes(bases, L):
    """gkm_idx_code of every window of `bases` (values 0..3), by start position"""
    bases = np.asarray(bases, np.uint32)
    nk = len(bases) - L + 1
    c = np.zeros(nk, np.uint32)
    for t in range(L):
        v = bases[t:t + nk]
        c |= ((v & 1) << base_bit(t, L, 0)) | ((v >> 1) << base_bit(t, L, 1))
    return c


def lex_to_code(L):
    """gkm_lt_lex_code for every lexicographic index (A, C, G, T = 0..3, first base most significant)"""
    lex = np.arange(4 ** L, dtype=np.uint32)
    c = np.zeros(4 ** L, np.uint32)
    for t in range(L):
        v = (lex >> (2 * (L - 1 - t))) & 3
        c |= ((v & 1) << base_bit(t, L, 0)) | ((v >> 1) << base_bit(t, L, 1))
    return c


def code_bases(L):
    """bases[u, t] = base t of the L-mer with code u"""
    u = np.arange(4 ** L, dtype=np.uint32)
    return np.stack([((u >> base_bit(t, L, 0)) & 1) | (((u >> base_bit(t, L, 1)) & 1) << 1) for t in range(L)], axis=1)


class Model:
    """what the table of a problem needs: per sequence its forward / reverse-complement bases and the weights of its
    windows (unit weights for kernel types 0..3)"""

    def __init__(self, problem, kernel_type, L, d, M=50, H=50.0):
        self.L, self.d, self.kernel_type = L, d, kernel_type
        self.w = problem.weights()
        self.fwd, self.rc, self.wt, self.wt_rc = [], [], [], []
        for i in range(problem.n):
            f, r = problem.codes(i)                  # 1..4 like gkm_data.seq
            f, r = f.astype(np.uint32) - 1, r.astype(np.uint32) - 1
            nk = len(f) - L + 1
            if kernel_type in (4, 5):
                a, b = capi.posweights(nk, kernel_type, M, H, lib=problem.lib)
            else:
                a = b = np.ones(nk, np.uint8)
            self.fwd.append(f)
            self.rc.append(r)
            self.wt.append(a.astype(np.float64))
            self.wt_rc.append(b.astype(np.float64))

    def postings(self, c):
        """(codes, weights) of column c in key-generation order: forward strand, then reverse complement, by window end"""
        return (np.concatenate((window_codes(self.fwd[c], self.L), window_codes(self.rc[c], self.L))),
                np.concatenate((self.wt[c], self.wt_rc[c])))

    def S(self, col0, alpha, norm):
        """S over the columns [col0, col0 + len(alpha)); norm[c] = |c| for every sequence of the problem"""
        S = np.zeros(4 ** self.L)
        for j, a in enumerate(alpha):
            codes, wts = self.postings(col0 + j)
            beta = np.float64(a) / np.float64(norm[col0 + j])
            np.add.at(S, codes, beta * wts)          # in order, one rounding per addition
        return S

    def longest_run(self, col0, ncols):
        """the most postings of one code: the longest sum S takes"""
        n = np.zeros(4 ** self.L, np.int64)
        for c in range(col0, col0 + ncols):
            np.add.at(n, self.postings(c)[0], 1)
        return int(n.max())

    def table(self, col0, alpha, norm):
        """T in code order"""
        return combine(transform(self.S(col0, alpha, norm), self.L, self.d), self.w)

    def forward(self, r):
        return window_codes(self.fwd[r], self.L), self.wt[r]

    def hist(self, r, c):
        """H_m(r, c), m = 0..d: the forward L-mers of r against the L-mers of both strands of c, weight products summed"""
        x, wx = self.forward(r)
        y, wy = self.postings(c)
        z = x[:, None] ^ y[None, :]
        m = sum(((z >> base_bit(t, self.L, 0)) | (z >> base_bit(t, self.L, 1))) & 1 for t in range(self.L))
        ww = wx[:, None] * wy[None, :]
        return np.array([ww[m == k].sum() for k in range(self.d + 1)])

    def scores(self, T, norm, rows, bias=0.0):
        out = np.zeros(len(rows))
        for i, r in enumerate(rows):
            x, wt = self.forward(r)
            s = np.cumsum(wt * T[x])[-1]             # sequential: 0 + p0 + p1 + ...
            out[i] = s / np.float64(norm[r]) + np.float64(bias)
        return out


def transform(S, L, d):
    """A[m] for m = 0..d: one step per base t = 0..L-1 on the groups of four codes that differ only in base t"""
    n = 4 ** L
    A = np.zeros((d + 1, n))
    A[0] = S
    for t in range(L):
        lo, hi = base_bit(t, L, 0), base_bit(t, L, 1)
        # view the codes as (above hi, bit hi, between, bit lo, below lo): base value v = (bit hi, bit lo)
        shape = (n >> (hi + 1), 2, 1 << (hi - lo - 1), 2, 1 << lo)
        V = [A[m].reshape(shape) for m in range(d + 1)]
        for m in range(d, 0, -1):
            lo_ = [V[m - 1][:, v >> 1, :, v & 1, :] for v in range(4)]
            for v in range(4):
                o = [u for u in range(4) if u != v]
                V[m][:, v >> 1, :, v & 1, :] = V[m][:, v >> 1, :, v & 1, :] + ((lo_[o[0]] + lo_[o[1]]) + lo_[o[2]])
    return A


def combine(A, w):
    T = np.zeros(A.shape[1])
    for m in range(A.shape[0]):
        T = T + w[m] * A[m]
    return T


def export(T, L):
    """T in lexicographic L-mer order"""
    return T[lex_to_code(L)]
