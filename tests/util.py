"""Shared helpers for the parity tests."""
import hashlib
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")

# float tolerance of the parity contract (BASELINE.json north_star: "within 1e-5
# relative float tolerance"; SURVEY.md 0.3 shows it can only be norm-wise because
# two builds of the reference itself differ by 2e-4 element-wise on stop-band
# outputs).  Norm-wise: max|d| <= RTOL * max|ref|.  Element-wise:
# |d| <= RTOL*|ref| + RTOL*max|ref|.
RTOL = 1e-5


def trunc4(x):
    """(int32)(x*10000): the reference's assert_cf32 semantics (test/utils.c:179)."""
    return (np.asarray(x, dtype=np.float32) * np.float32(10000)).astype(np.int32)


def digest(a):
    """First 16 hex digits of the SHA-256 of an array's bytes: bit-for-bit comparison with
    a stored output without storing the output itself."""
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


def reference_outputs():
    """What the reference, compiled unmodified, computed for the inputs the tests generate
    (recorded by tests/golden/record_reference_outputs.py): digests of bit-exact outputs
    (JSON) and samples of outputs compared within a tolerance (NPZ)."""
    with open(os.path.join(GOLDEN, "reference_outputs.json")) as f:
        digests = json.load(f)
    with np.load(os.path.join(GOLDEN, "reference_outputs.npz")) as z:
        samples = {k: z[k] for k in z.files}
    return digests, samples


def harness_blocks(n_blocks, block_bytes=262144):
    """The input blocks of oracle/ref_server_harness.c: one xorshift64 byte stream."""
    m = (1 << 64) - 1
    s = 0x9E3779B97F4A7C15
    out = bytearray(n_blocks * block_bytes)
    for i in range(len(out)):
        s ^= (s << 13) & m
        s ^= s >> 7
        s ^= (s << 17) & m
        out[i] = s & 0xFF
    return np.frombuffer(bytes(out), dtype=np.uint8).reshape(n_blocks, block_bytes)


def ramp(fmt, offset, n):
    """Input generators of the reference's tests (test/utils.c:137-165)."""
    i = np.arange(n, dtype=np.int64) + offset
    if fmt == "cu8":
        return (i & 0xFF).astype(np.uint8)
    if fmt == "cs8":
        return (i & 0xFF).astype(np.uint8).view(np.int8)
    return ((i & 0xFFFF).astype(np.uint16).view(np.int16) - np.int16(n // 2)).astype(np.int16)


def rand_block(rng, fmt, n):
    if fmt == "cs16":
        return rng.integers(-8192, 8192, n, dtype=np.int16)
    if fmt == "cs8":
        return rng.integers(-128, 128, n, dtype=np.int8)
    return rng.integers(0, 256, n, dtype=np.uint8)


def assert_cf32_close(got, ref, what=""):
    got = np.asarray(got, dtype=np.complex64)
    ref = np.asarray(ref, dtype=np.complex64)
    assert got.shape == ref.shape, f"{what}: output count {got.shape} != {ref.shape}"
    if ref.size == 0:
        return 0.0
    d = np.abs(got.astype(np.complex128) - ref.astype(np.complex128))
    scale = float(np.max(np.abs(ref)))
    if scale == 0.0:
        assert float(d.max()) == 0.0, f"{what}: reference is all zero, got max {d.max()}"
        return 0.0
    worst = int(np.argmax(d))
    assert d.max() <= RTOL * scale, (f"{what}: norm-wise error {d.max() / scale:.3e} > {RTOL} at k={worst} "
                                     f"(got {got[worst]}, ref {ref[worst]})")
    bound = RTOL * np.abs(ref) + RTOL * scale
    bad = np.nonzero(d > bound)[0]
    assert bad.size == 0, f"{what}: {bad.size} outputs beyond element-wise bound, first k={bad[0]}"
    return float(d.max() / scale)


def oracle_stream(oracles, fmt, blocks, keep=None, workers=None, renorm=True):
    """Run every oracle filter over the whole block sequence (in order: the filters
    carry history and phase) on a thread pool -- ctypes releases the GIL while the C
    oracle runs.  Returns out[client][block] for the block indices in `keep` (all
    blocks when None); other entries are None."""
    import os
    from concurrent.futures import ThreadPoolExecutor
    keep = set(range(len(blocks))) if keep is None else set(keep)
    workers = workers or min(len(oracles), max(1, (os.cpu_count() or 2) - 1), 64)

    def run(o):
        res = []
        for b, x in enumerate(blocks):
            y = o.process_cf32(fmt, x, renorm=renorm)
            res.append(y if b in keep else None)
        return res

    with ThreadPoolExecutor(max_workers=workers) as ex:
        return list(ex.map(run, oracles))
