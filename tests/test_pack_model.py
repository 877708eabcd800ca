"""CPU tier: the packed problem image of the host packer (gkm_seq.c: gkm_pack_problem, which every CPU emulator runs)
against the numpy model of the image (pack_model.py).  The host packer applies the rule of gkm_pack.h, which the device
packer (gkm_device.cu: gkm_pack_kernel) includes verbatim; the GPU tier holds the device image to the same model on the
same cases (test_gpu_abi.py::test_device_packing_equals_model)."""
import ctypes
import os

import numpy as np
import pytest

import pack_model
from gkmqc_b200 import capi


@pytest.fixture(scope="module")
def abi_emu():
    import __graft_entry__ as ge
    lib = ctypes.CDLL(os.environ.get("GKM_ABI_EMU_LIB") or ge.build_abi_emulator())
    capi._declare(lib)
    return lib


def check(lib, kernel_type, L, M, H, seqs):
    with capi.Problem(*pack_model.problem_args(kernel_type, L, M, H), lib=lib) as P:
        P.add_many(seqs)
        planes, wend = P.image()
    want_planes, want_wend = pack_model.image(seqs, L, kernel_type, M, H, lib)
    assert planes.shape == want_planes.shape
    for plane, what in enumerate(("code bit 0", "code bit 1", "window ends")):
        assert np.array_equal(planes[:, plane], want_planes[:, plane]), what
    if kernel_type in (4, 5):
        assert np.array_equal(wend, want_wend), "positional weights by window end"
    else:
        assert wend is None
    return wend


@pytest.mark.parametrize("kernel_type,L,M,H", pack_model.PARAMS)
def test_host_packing_equals_model(kernel_type, L, M, H, abi_emu):
    wend = check(abi_emu, kernel_type, L, M, H, pack_model.sequences(L))
    if wend is not None:
        assert wend.max() == (M if M < 255 else 247)  # M = 255: the centre weight 256 wraps to 0 in the reference's u_int8_t


@pytest.mark.parametrize("seed", range(8))
def test_host_packing_equals_model_generated(seed, abi_emu):
    """random parameters, lengths from L to past a word boundary, and any byte: A, C, G, T in either case, the other
    255 - 8 byte values counting as A"""
    rng = np.random.default_rng(seed)
    kernel_type = int(rng.choice([0, 2, 4, 5]))
    L = int(rng.integers(2, 17))
    M, H = int(rng.integers(1, 256)), float(rng.uniform(1.0, 100.0))
    seqs = []
    for _ in range(int(rng.integers(1, 40))):
        ln = int(rng.integers(L, 300))
        s = np.frombuffer(b"ACGTacgt", np.uint8)[rng.integers(0, 8, ln)]
        other = rng.random(ln) < 0.1
        s[other] = rng.integers(0, 256, int(other.sum()))
        seqs.append(s.tobytes())
    check(abi_emu, kernel_type, L, M, H, seqs)
