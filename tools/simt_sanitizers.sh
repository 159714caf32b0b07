#!/bin/bash
# The emulated-kernel suites (tests/test_kernel_simt.py, and the routing / gathered-quantiser cases of tests/test_moe_prefill_simt.py) under AddressSanitizer: the wide path's kernel SOURCE runs on the CPU (tests/hostsim/simt.h) with every
# global / "shared" memory access bounds-checked — weight rows, activation columns, outputs (numpy buffers on the ASan heap) and the static __shared__ arrays.
# Then the same under ThreadSanitizer: the emulation's only synchronisation is __syncthreads / warp shuffles, so a shared-memory hand-over between
# threads of a block that lacks a barrier shows up as a data race.
# No GPU needed.  Expected: all tests pass, no AddressSanitizer report, no "ThreadSanitizer: data race".
set -e
cd "$(dirname "$0")/.."
SIM=tests/hostsim
LIBS="kernsim moesim"
for l in $LIBS; do cp $SIM/lib$l.so /tmp/lib${l}_plain.so 2>/dev/null || true; done
for l in $LIBS; do
    g++ -O1 -g -std=c++20 -fPIC -shared -pthread -ffp-contract=off -w -fsanitize=address -fno-omit-frame-pointer -I/usr/local/cuda/include -x c++ $SIM/$l.cpp -o $SIM/lib$l.so
    touch $SIM/lib$l.so
done
ASAN_OPTIONS=detect_leaks=0:halt_on_error=1 LD_PRELOAD=$(gcc -print-file-name=libasan.so) python -m pytest tests/test_kernel_simt.py tests/test_moe_prefill_simt.py -k "not workspace" -x -q -p no:cacheprovider
rc=$?
for l in $LIBS; do
    g++ -O1 -g -std=c++20 -fPIC -shared -pthread -ffp-contract=off -w -fsanitize=thread -I/usr/local/cuda/include -x c++ $SIM/$l.cpp -o $SIM/lib$l.so
    touch $SIM/lib$l.so
done
TSAN_OPTIONS="halt_on_error=0 report_signal_unsafe=0 exitcode=0" LD_PRELOAD=$(gcc -print-file-name=libtsan.so) python -m pytest tests/test_kernel_simt.py tests/test_moe_prefill_simt.py -k "not workspace" -x -q -p no:cacheprovider > /tmp/simt_tsan.log 2>&1 || rc=1
tail -1 /tmp/simt_tsan.log
if grep -q "ThreadSanitizer: data race" /tmp/simt_tsan.log; then echo "data races reported: see /tmp/simt_tsan.log"; rc=1; else echo "ThreadSanitizer: no data race"; fi
for l in $LIBS; do [ -f /tmp/lib${l}_plain.so ] && cp /tmp/lib${l}_plain.so $SIM/lib$l.so && touch $SIM/lib$l.so; done
exit $rc
