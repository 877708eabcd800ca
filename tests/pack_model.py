"""The packed problem image restated in numpy from the letters: what the device packer (gkm_device.cu: gkm_pack_kernel) and
the host packer of the CPU emulators (gkm_seq.c: gkm_pack_problem) must both build from gkm_pack.h.

Per sequence one circular string of 32 W positions, W = ceil(2 maxlen / 32): the forward codes at [0, len), the mirrored
complement at [len, 2 len) (libgkm.c:878-888), zero padding behind.  planes[i] = (code bit 0, code bit 1, E), position j
at bit j % 32 of word j // 32; E marks the positions at which an L-mer of either strand ends.  wend[i][j] = weight of that
L-mer, taken per position from gkm_calc_posweights (capi.posweights: wt for the forward strand, wt_rc for the reverse
one), not from the distance table the packers index."""
import numpy as np

from conftest import random_seqs
from gkmqc_b200 import capi

# A, C, G, T in either case -> 0..3; every other byte counts as A (libgkm.c:864-875)
LETTER_CODE = np.zeros(256, np.uint8)
for _code, _letters in enumerate((b"Aa", b"Cc", b"Gg", b"Tt")):
    for _ch in _letters:
        LETTER_CODE[_ch] = _code

# (kernel_type, L, M, H): unweighted, weighted, weighted at M = 255 (the centre weight wraps to 0), and L = 3 at M = 1
PARAMS = [(2, 11, 50, 50.0), (4, 11, 50, 50.0), (5, 10, 255, 20.0), (4, 3, 1, 3.0)]


def problem_args(kernel_type, L, M, H):
    """Problem(...) arguments of a parameter set: k and d do not reach the image"""
    k = min(L, 7)
    return kernel_type, L, k, min(3, L - k), M, H, 1.0


def sequences(L):
    """ragged random rows, rows at the word boundaries and at the longest length the engine holds, lower case and
    letters that are not nucleotides"""
    seqs = [s.encode() for s in random_seqs(257, 400, seed=11, ragged=True)]
    rng = np.random.default_rng(5)
    for ln in (L, L + 1, 31, 32, 33, 63, 64, 65, 96, 1024, 2046, 2047):
        if ln >= L:
            seqs.append(np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, ln)].tobytes())
    seqs[3] = b"acgtNNacgtRYacgtacgt" + seqs[3]
    return seqs


def image(seqs, L, kernel_type, M, H, lib=None):
    """(planes [n, 3, W] uint32, wend [n, 32 W] uint8 or None) of the rows `seqs` (bytes)"""
    W = (2 * max(len(s) for s in seqs) + 31) // 32
    planes = np.zeros((len(seqs), 3, W), np.uint32)
    wend = np.zeros((len(seqs), 32 * W), np.uint8) if kernel_type in (4, 5) else None
    for i, s in enumerate(seqs):
        ln = len(s)
        fwd = LETTER_CODE[np.frombuffer(s, np.uint8)]
        code = np.zeros(32 * W, np.uint8)
        code[:ln] = fwd
        code[ln:2 * ln] = 3 - fwd[::-1]
        end = np.zeros(32 * W, bool)
        end[L - 1:ln] = True
        end[ln + L - 1:2 * ln] = True
        bits = np.stack([code & 1, code >> 1, end]).astype(np.uint64).reshape(3, W, 32)
        planes[i] = (bits << np.arange(32, dtype=np.uint64)).sum(axis=2)
        if wend is not None:
            wt, wt_rc = capi.posweights(ln - L + 1, kernel_type, M, H, lib)
            wend[i, L - 1:ln] = wt
            wend[i, ln + L - 1:2 * ln] = wt_rc
    return planes, wend
