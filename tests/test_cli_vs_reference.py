"""CPU tier: the stand-alone CLI (gkmqc_b200/csrc/gkmkern_cli.c, SURVEY.md 8f/f3) against the reference's own `gkmkern`
(src/gkmkern_main.c, compiled unmodified into oracle/_ref/gkmkern).  The product's CLI source is linked here against the
ABI emulator library (test infrastructure: host code of the product over a host stand-in of the device layer); the shipped
gkmqc_b200/bin/gkmkern links the CUDA library and is covered by tests/test_gpu_cli.py.

Same positional arguments, same default parameters (EST_TRUNC, L=10 k=6 d=3: gkmkern_main.c:99-107), same output format
("%e\\t" per entry, "1.0\\t" on the diagonal: gkmkern_main.c:221-228): the output FILES must be equal byte for byte when
the number of sequences is a multiple of four; otherwise the reference silently drops the last N mod 4 rows
(gkmkern_main.c:58,221) and the product writes them all."""
import os
import subprocess

import numpy as np
import pytest

import pyoracle
from conftest import load_golden, random_seqs, write_fasta

REF_CLI = os.path.join(pyoracle.REF_DIR, "gkmkern")
needs_ref_cli = pytest.mark.skipif(not os.path.exists(REF_CLI), reason="oracle/_ref/gkmkern (the compiled reference CLI) is not here")


@pytest.fixture(scope="module")
def cli():
    import __graft_entry__ as ge
    return ge.build_cli_emulator()


def files(tmp_path, n, seed):
    seqs = random_seqs(n, 160, seed=seed, ragged=True)
    seqs[1] = seqs[0]                       # a duplicate
    seqs[2] = seqs[2].lower()               # lower case counts like upper case (libgkm.c:864-875)
    pos, neg = tmp_path / "pos.fa", tmp_path / "neg.fa"
    write_fasta(str(pos), seqs[: n // 2], "p")
    write_fasta(str(neg), seqs[n // 2:], "n")
    return str(pos), str(neg)


@needs_ref_cli
@pytest.mark.parametrize("n", [24, 8])
def test_same_output_file_as_the_reference_cli(tmp_path, cli, n):
    pos, neg = files(tmp_path, n, seed=n)
    ref_out, our_out = str(tmp_path / "ref.tsv"), str(tmp_path / "ours.tsv")
    assert subprocess.run([REF_CLI, pos, neg, ref_out], stdout=subprocess.DEVNULL).returncode == 0
    assert subprocess.run([cli, "-v", "0", pos, neg, our_out], stdout=subprocess.DEVNULL).returncode == 0
    a, b = open(ref_out, "rb").read(), open(our_out, "rb").read()
    assert a == b
    assert a.count(b"\n") == n


@needs_ref_cli
def test_rows_the_reference_cli_drops(tmp_path, cli):
    pos, neg = files(tmp_path, 26, seed=3)
    ref_out, our_out = str(tmp_path / "ref.tsv"), str(tmp_path / "ours.tsv")
    assert subprocess.run([REF_CLI, pos, neg, ref_out], stdout=subprocess.DEVNULL).returncode == 0
    assert subprocess.run([cli, "-v", "0", pos, neg, our_out], stdout=subprocess.DEVNULL).returncode == 0
    a, b = open(ref_out, "rb").read().splitlines(), open(our_out, "rb").read().splitlines()
    assert len(a) == 24 and len(b) == 26 and b[:24] == a
    assert all(line.endswith(b"1.0\t") and line.count(b"\t") == i + 1 for i, line in enumerate(b))


def test_options_reach_the_engine(tmp_path, cli):
    """-t -l -k -d -M -H and -p 17 (loss-free doubles) / -b (binary): the values are those the reference's gkm_main_pywrapper
    returned for the same parameters and files (tests/golden, written from the unmodified reference by oracle/gen_golden.py);
    the two stored sets move -t -M -H and -l -k -d off the CLI's defaults"""
    txt, binf = str(tmp_path / "o.tsv"), str(tmp_path / "o.bin")
    for name in ("mix_t4_L10k6d3_M255", "mix_t2_L8k4d4"):
        g, cfg, pos, neg = load_golden(name)
        K, n = g["kmat"], len(g["lens"])
        common = ["-v", "0", "-t", str(cfg["kernel_type"]), "-l", str(cfg["L"]), "-k", str(cfg["k"]), "-d", str(cfg["d"]),
                  "-M", str(cfg["M"]), "-H", repr(cfg["H"])]
        assert subprocess.run([cli] + common + ["-p", "17", pos, neg, txt], stdout=subprocess.DEVNULL).returncode == 0
        assert subprocess.run([cli] + common + ["-b", pos, neg, binf], stdout=subprocess.DEVNULL).returncode == 0
        rows = [np.array([float(x) for x in line.split("\t")[:-1]]) for line in open(txt).read().splitlines()]
        assert len(rows) == n
        raw = open(binf, "rb").read()
        assert np.frombuffer(raw[:4], np.int32)[0] == n
        flat = np.frombuffer(raw[4:], np.float64)
        at = 0
        for a in range(n):
            assert np.array_equal(rows[a][:a], K[a, :a]) and rows[a][a] == 1.0, (name, a)
            assert np.array_equal(flat[at:at + a], K[a, :a]), (name, a)
            at += a
        assert at == len(flat)
    # what the gate refuses is refused here too, with the reference's message
    r = subprocess.run([cli, "-l", "13", pos, neg, txt], capture_output=True, text=True)
    assert r.returncode == 0 or "L" in r.stderr          # L = 13..16 is the CLI's documented extension
    r = subprocess.run([cli, "-l", "6", "-k", "5", "-d", "3", pos, neg, txt], capture_output=True, text=True)
    assert r.returncode == 1 and "d > L - k" in r.stderr
