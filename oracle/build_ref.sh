#!/bin/bash
# oracle/build_ref.sh -- TEST INFRASTRUCTURE.  Builds oracle/_ref/ from the UNMODIFIED
# reference sources where they lie under $REF_DIR (never copied into this repo; the one
# scratch copy, _ref/patched/, is a build product and git-ignored like all of _ref/).
# Called by oracle/Makefile; see the table there for what each output is.
set -e
REF_DIR="${REF_DIR:-/root/reference}"
CC="${CC:-gcc}"
cd "$(dirname "$0")"
if [ ! -f "$REF_DIR/src/xlating.c" ]; then
  echo "REF_DIR=$REF_DIR not present: keeping prebuilt oracle/_ref (if any)"
  exit 0
fi
mkdir -p _ref
R="$REF_DIR"
REF_SRC="$R/src/xlating.c $R/src/lpf.c"
UNITY_INC="-I$R/test/unity-2.5.2/src -I$R/test -I$R/src"
UNITY_SRC="$R/test/unity-2.5.2/src/unity.c"
STRICT="-std=gnu11 -O2 -ffp-contract=off"
FAST="-std=gnu11 -O3 -DNDEBUG -ffast-math"
B200_LIB=../sdr-server_b200/lib/libxlating_b200.so
B200_LINK="-L../sdr-server_b200/lib -lxlating_b200 -Wl,-rpath,\$ORIGIN/../../sdr-server_b200/lib -lm"
HOST=../sdr-server_b200/host

# --- the reference's DSP unit as shared libraries (parity target + CPU timing) ---
$CC -std=c11 -O2 -ffp-contract=off -fPIC -shared -I$R/src -o _ref/libref_strict.so $REF_SRC -lm
$CC $FAST -fPIC -shared -I$R/src -o _ref/libref_release.so $REF_SRC -lm
$CC $FAST -mavx2 -mfma -fPIC -shared -I$R/src -o _ref/libref_avx.so $REF_SRC -lm
# --- pinned thread-per-client CPU timing in C, one binary per flag set ---
$CC $FAST -pthread -I$R/src -o _ref/ref_cpu_bench_release ref_cpu_bench.c $REF_SRC -lm
$CC $FAST -mavx2 -mfma -pthread -I$R/src -o _ref/ref_cpu_bench_avx ref_cpu_bench.c $REF_SRC -lm
$CC $FAST -march=x86-64-v3 -pthread -I$R/src -o _ref/ref_cpu_bench_v3 ref_cpu_bench.c $REF_SRC -lm
$CC $FAST -march=x86-64-v4 -pthread -I$R/src -o _ref/ref_cpu_bench_v4 ref_cpu_bench.c $REF_SRC -lm
# --- the reference's own programs on the reference's own sources (prove the stand-ins) ---
$CC $FAST -mavx2 -mfma -I$R/src -o _ref/perf_xlating_ref $R/test/perf_xlating.c $REF_SRC -lm
$CC $STRICT $UNITY_INC -o _ref/test_xlating_ref $R/test/test_xlating.c ref_test_support.c $UNITY_SRC $REF_SRC -lz -lm
$CC $STRICT $UNITY_INC -o _ref/test_lpf_ref $R/test/test_lpf.c $UNITY_SRC $R/src/lpf.c -lm
$CC $STRICT $UNITY_INC -pthread -o _ref/test_queue_ref $R/test/test_queue.c $UNITY_SRC $R/src/queue.c
HARNESS="-include unistd.h -I$R/src -I../include -pthread ref_server_harness.c $R/src/dsp_worker.c"
$CC $STRICT -o _ref/server_harness_ref $HARNESS $R/src/queue.c $REF_SRC -lz -lm
$CC $FAST -mavx2 -mfma -o _ref/server_harness_ref_avx $HARNESS $R/src/queue.c $REF_SRC -lz -lm
# the reference's whole server integration test (test/test_tcp_server.c, 11 tests) with its
# real tcp_server.c / dsp_worker.c / queue.c / sdr_device.c / device wrappers / client / mocks;
# stand-ins only for what this image lacks: vendor headers (stubs/), libconfig (ref_config_standin.c),
# libpng (ref_test_support.c instead of test/utils.c)
SERVER_TEST="-include unistd.h -Istubs $UNITY_INC -pthread $R/test/test_tcp_server.c $R/test/rtlsdr_lib_mock.c \
  $R/test/airspy_lib_mock.c $R/test/hackrf_lib_mock.c $R/src/sdr_device.c $R/src/sdr/rtlsdr_device.c \
  $R/src/sdr/airspy_device.c $R/src/sdr/hackrf_device.c $R/src/client/tcp_client.c ref_config_standin.c \
  ref_test_support.c $UNITY_SRC"
$CC $STRICT -w -o _ref/test_tcp_server_ref $SERVER_TEST $R/src/tcp_server.c $R/src/dsp_worker.c $R/src/queue.c $REF_SRC -lz -lm
cp "$R/test/resources/tcp_server.config" _ref/tcp_server.config
# --- the pinned-block queue (sdr-server_b200/host/queue_pinned.c) under the reference's own queue test ---
$CC $STRICT $UNITY_INC -I../include -DXL_QUEUE_PAGEABLE -pthread -o _ref/test_queue_pageable $R/test/test_queue.c $UNITY_SRC $HOST/queue_pinned.c

# --- the reference's src/ as it is (tests compare our headers with it and apply the patch to it) ---
rm -rf _ref/src
cp -r "$R/src" _ref/src
chmod -R u+w _ref/src  # the reference may be read-only; its copies are patched
# --- integration/cuda_cf32.patch applied to a scratch copy of the reference's src/ ---
rm -rf _ref/patched
mkdir -p _ref/patched
cp -r "$R/src" _ref/patched/src
chmod -R u+w _ref/patched/src
patch -s -p1 -d _ref/patched < ../integration/cuda_cf32.patch
P=_ref/patched/src
# the patched control plane still parses (libconfig is absent: syntax only for config.c)
$CC -std=gnu11 -fsyntax-only -I../include -Istubs/libconfig $P/config.c

if [ -f "$B200_LIB" ]; then
  # --- the reference's own programs, unmodified, on libxlating_b200.so ---
  $CC -std=gnu11 -O2 -o _ref/perf_xlating_b200 $R/test/perf_xlating.c $B200_LINK
  $CC -std=gnu11 -O2 $UNITY_INC -o _ref/test_xlating_b200 $R/test/test_xlating.c ref_test_support.c $UNITY_SRC -lz $B200_LINK
  $CC -std=gnu11 -O2 $UNITY_INC -o _ref/test_lpf_b200 $R/test/test_lpf.c $UNITY_SRC $B200_LINK
  $CC -std=gnu11 -O2 -o _ref/server_harness_b200 $HARNESS $R/src/queue.c -lz $B200_LINK
  $CC -std=gnu11 -O2 -o _ref/server_harness_b200_pinnedq $HARNESS $HOST/queue_pinned.c -lz $B200_LINK
  $CC -std=gnu11 -O2 -w -o _ref/test_tcp_server_b200 $SERVER_TEST $R/src/tcp_server.c $R/src/dsp_worker.c $R/src/queue.c -lz $B200_LINK
  $CC $STRICT $UNITY_INC -I../include -pthread -o _ref/test_queue_pinned $R/test/test_queue.c $UNITY_SRC $HOST/queue_pinned.c $B200_LINK
  # --- the PATCHED reference (cpu_optimization = CUDA_CF32 -> batch ABI) ---
  PSERVER_TEST="${SERVER_TEST//$R\/src\//$P/}"
  PSERVER_TEST="${PSERVER_TEST//-I$R\/src/-I$P}"
  # CPU modes of the patched tree on the reference's own xlating.c: the patch must not change them
  $CC $STRICT -w -DXL_HAVE_CUDA_CF32 -I../include -o _ref/test_tcp_server_patched_ref $PSERVER_TEST $P/tcp_server.c $P/dsp_worker.c $P/queue.c $P/xlating.c $P/lpf.c -lz $B200_LINK
  # CUDA_CF32 (XL_TEST_CPU_OPTIMIZATION=CUDA_CF32 selects it in the config stand-in)
  $CC -std=gnu11 -O2 -w -DXL_HAVE_CUDA_CF32 -I../include -o _ref/test_tcp_server_patched_b200 $PSERVER_TEST $P/tcp_server.c $P/dsp_worker.c $P/queue.c -lz $B200_LINK
  $CC -std=gnu11 -O2 -DHARNESS_CUDA_CF32 -include unistd.h -I$P -I../include -pthread -o _ref/server_harness_patched_b200 ref_server_harness.c $P/dsp_worker.c $P/queue.c -lz $B200_LINK
fi
echo "built oracle/_ref from $REF_DIR"
