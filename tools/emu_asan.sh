#!/bin/bash
# Memory check of the device step code without a GPU: the kernel source (csrc/*.cuh) compiled for the host SIMT
# emulator with AddressSanitizer and exact-size shared-memory stand-ins, driven by the emulator parity tests.
set -e
cd "$(dirname "$0")/.."
sed 's/env_words + 64/env_words/; s/4 \* img.dm.nprobe + 4/4 * ((img.dm.nprobe + 3) \& ~3)/' tests/emu/emu_lib.cpp > tests/emu/_asan_tmp.cpp
cp tests/emu/libmjb_emu.so /tmp/libmjb_emu_backup.so 2>/dev/null || true
g++ -O1 -g -std=c++17 -fPIC -shared -fsanitize=address -Wno-unknown-pragmas -o tests/emu/libmjb_emu.so tests/emu/_asan_tmp.cpp
rm tests/emu/_asan_tmp.cpp
# (the compile-refusal tests are left out: a C++ exception thrown by the uninstrumented libmjb.so aborts under the preloaded runtime)
ASAN_OPTIONS=detect_leaks=0:detect_stack_use_after_return=0 LD_PRELOAD=$(g++ -print-file-name=libasan.so) \
  python -m pytest tests/test_emu_parity.py "tests/test_ext_sensors.py" -k "not refusals" -m "not gpu" -x -q || rc=$?
rm -f tests/emu/libmjb_emu.so   # rebuilt without the sanitizer on the next test run
exit ${rc:-0}
