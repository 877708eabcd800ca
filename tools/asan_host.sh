#!/bin/sh
# The host C of the library (FASTA reader, coding, host packer, weights, chunk planner, index cost model, and the
# reference-ABI shim gkm_capi.c over the host stand-in of the device layer) and the CPU emulators of the index variant
# and of the L-mer table and its substitutions
# under AddressSanitizer + UndefinedBehaviorSanitizer, driven by the CPU test tier.
# The CUDA objects cannot be sanitised this way (nvcc, static cudart), and compute-sanitizer is closed on this GPU pool
# (tools/sanitize_target.py is the command it would run): the device code's addressing rules are checked on the CPU by the
# emulators this script runs.  The bit-sliced emulator is compiled plain: its templates take minutes under ASan.
set -e
cd "$(dirname "$0")/.."
B=build/asan
C=gkmqc_b200/csrc
SAN="-fsanitize=address,undefined -fno-omit-frame-pointer -g -O1 -fPIC"
mkdir -p $B
for f in gkm_seq gkm_weights gkm_log gkm_sched gkm_options gkm_index_host gkm_capi; do
    gcc -std=gnu11 -ffp-contract=off $SAN -c $C/$f.c -o $B/$f.o
done
g++ -std=c++17 $SAN -c tests/emu/index_emu.cc -o $B/index_emu.o
g++ -std=c++17 $SAN -ffp-contract=off -c tests/emu/lmer_table_emu.cc -o $B/lmer_table_emu.o
g++ -std=c++17 $SAN -ffp-contract=off -c tests/emu/lmer_subst_emu.cc -o $B/lmer_subst_emu.o
g++ -std=c++17 $SAN -ffp-contract=off -c tests/emu/dev_stub.cc -o $B/dev_stub.o
g++ -std=c++17 -O1 -fPIC -ffp-contract=off -c tests/emu/diag_emu.cc -o $B/diag_emu.o
HOSTO="$B/gkm_seq.o $B/gkm_weights.o $B/gkm_log.o $B/gkm_sched.o $B/gkm_options.o $B/gkm_index_host.o"
g++ -shared -fsanitize=address,undefined -o $B/libgkm_emu_asan.so $B/diag_emu.o $B/index_emu.o $B/lmer_table_emu.o $B/lmer_subst_emu.o $HOSTO -lm -lpthread
g++ -shared -fsanitize=address,undefined -o $B/libgkm_abi_emu_asan.so $B/diag_emu.o $B/dev_stub.o $B/gkm_capi.o $HOSTO -lm -lpthread
LIB=$PWD/$B/libgkm_emu_asan.so
# leaks are not checked: the interpreter itself never frees most of what it allocates
LD_PRELOAD=$(gcc -print-file-name=libasan.so) ASAN_OPTIONS=detect_leaks=0 UBSAN_OPTIONS=print_stacktrace=1:halt_on_error=1 \
GKM_PYLIB=$LIB GKM_EMU_LIB=$LIB GKM_ABI_EMU_LIB=$PWD/$B/libgkm_abi_emu_asan.so python -m pytest -q -x -m "not gpu" \
    tests/test_abi_on_emulator.py tests/test_abi_vs_reference.py tests/test_pywrapper_vs_reference.py tests/test_fasta_fuzz.py tests/test_sched_properties.py tests/test_posweights_properties.py \
    tests/test_host_logic.py tests/test_index_host.py tests/test_emu_bitslice.py tests/test_lmer_table_model.py tests/test_lmer_subst_model.py \
    tests/test_pack_model.py \
    --deselect tests/test_host_logic.py::test_library_exports_every_declared_symbol \
    --deselect tests/test_host_logic.py::test_copy_threads_policy \
    --deselect tests/test_host_logic.py::test_compute_fails_loudly_without_gpu "$@"
