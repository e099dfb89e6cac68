# usage: bash tools/run_emu_sanitized.sh   -- the host build of the kernel sources (tests/simt_emu) under AddressSanitizer +
# UndefinedBehaviorSanitizer: the emulator suites, with libasan (and libstdc++, whose __cxa_throw ASan must find at start-up:
# the oracle throws and catches) preloaded into the Python process.  compute-sanitizer is closed on the GPU pool; this is
# how the indexing of the kernels (ragged tiles, idle slots, fallbacks, the launch-overlap counters) is checked.
ASAN=$(/usr/bin/g++ -print-file-name=libasan.so)
STDCPP=$(/usr/bin/g++ -print-file-name=libstdc++.so)
rm -f /tmp/ukfb_asan.* /tmp/ukfb_ubsan.*
UKFB_EMU_SANITIZE=1 LD_PRELOAD="$ASAN $STDCPP" \
  ASAN_OPTIONS=detect_leaks=0:halt_on_error=1:log_path=/tmp/ukfb_asan \
  UBSAN_OPTIONS=halt_on_error=1:print_stacktrace=1:log_path=/tmp/ukfb_ubsan \
  python -m pytest tests/test_emu_lane_kernels.py tests/test_emu_parity.py tests/test_gate.py tests/test_events.py \
    tests/test_so3_kernels.py tests/test_emu_indexed.py tests/test_emu_checkpoint.py -x -q -m "not gpu" -p no:cacheprovider
rc=$?
ls /tmp/ukfb_asan.* /tmp/ukfb_ubsan.* 2>/dev/null && { echo "sanitizer reports written"; rc=1; }
exit $rc
