#!/usr/bin/env python3
"""Record what the reference computes for the inputs of the tests that compare with it
into tests/golden/reference_outputs.json (digests of outputs compared bit for bit) and
tests/golden/reference_outputs.npz (samples of outputs compared within a tolerance).

Needs oracle/_ref/ (the reference's sources compiled unmodified by `make -C oracle` where
the reference is present) and runs without a GPU.  The files it writes are committed and
are what the tests read:
  tests/test_oracle.py              the restatement against the reference's DSP unit
  tests/test_reference_programs.py  the restatement against the files the reference's own
                                    dsp_worker threads write (oracle/ref_server_harness.c)
"""
import json
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.dirname(HERE)]

from oracle import pyoracle as po  # noqa: E402
import test_oracle as t  # noqa: E402
import test_reference_programs as trp  # noqa: E402
from util import digest  # noqa: E402


def main():
    for flavor in ("strict", "release", "avx"):
        if not po.ref_available(flavor):
            raise SystemExit(f"oracle/_ref/libref_{flavor}.so not built (make -C oracle with the reference present)")
    out = {"_source": "dernasherbrezon/sdr-server src/xlating.c + src/lpf.c compiled unmodified (oracle/_ref)",
           "_digest": "first 16 hex digits of the SHA-256 of the output's bytes (tests/util.py digest)"}

    out["lpf"] = {t.case_key(*c): digest(po.ref_lpf_design(1.0, *c)) for c in t.LPF_CASES}

    out["stream"] = {}
    for fs, rate, tw, center in t.STREAM_CASES:
        taps = po.lpf_design(1.0, fs, rate // 2, tw)
        for fmt in t.STREAM_FMTS:
            f = po.RefFilter(fs // rate, taps, center, fs, 40000)
            q = po.RefFilter(fs // rate, taps, center, fs, 40000)
            out["stream"][t.case_key(fmt, fs, rate, tw, center)] = [
                [digest(f.process_cf32(fmt, x)), digest(q.process_q15(fmt, x))] for x in t.stream_inputs(fmt)]

    out["random_shapes"] = {}
    for seed in t.RANDOM_SEEDS:
        shapes = []
        for T, D, fs, center, taps, max_in, fmt, xs in t.random_shapes(seed):
            f = po.RefFilter(D, taps, center, fs, max_in)
            q = po.RefFilter(D, taps, center, fs, max_in)
            shapes.append([[digest(f.process_cf32(fmt, x)), digest(q.process_q15(fmt, x))] for x in xs])
        out["random_shapes"][str(seed)] = shapes

    # the reference's own dsp_worker threads (oracle/ref_server_harness.c, strict build)
    clients, blocks = trp.HARNESS_ON_REFERENCE
    with tempfile.TemporaryDirectory() as tmp:
        r = trp.run_harness("server_harness_ref", clients, blocks, 8, tmp, "rtl", "dump")
        assert r.returncode == 0, r.stderr[-400:]
        raw = np.fromfile(os.path.join(tmp, "input.raw"), dtype=np.uint8)
        outs = [digest(np.fromfile(os.path.join(tmp, f"{c}.cf32"), dtype=np.complex64)) for c in range(clients)]
    out["server_harness"] = {"clients": clients, "blocks": blocks, "input": digest(raw), "outputs": outs}

    samples = {}
    rng = np.random.default_rng(20261017)
    seed, fs, rate, tw, center, n, n_blocks = t.NORM_WISE
    taps = po.lpf_design(1.0, fs, rate // 2, tw)
    strict = po.RefFilter(fs // rate, taps, center, fs, n, "strict")
    release = po.RefFilter(fs // rate, taps, center, fs, n, "release")
    avx = po.RefFilter(fs // rate, taps, center, fs, n, "avx")
    idx, rel, av = [], [], []
    for x in t.cu8_blocks(seed, n, n_blocks):
        s, a, b = (f.process_cf32("cu8", x) for f in (strict, release, avx))
        # keep the 32 outputs of the block where the fast builds differ most from the strict
        # one in absolute terms and the 32 where they differ most relative to the output:
        # the worst cases of both the norm-wise and the element-wise comparison
        d = np.maximum(np.abs(a - s), np.abs(b - s)).astype(np.float64)
        r = np.where(np.abs(s) > 0, d / np.maximum(np.abs(s), 1e-30), 0.0)
        i = np.unique(np.concatenate([np.argsort(d)[-32:], np.argsort(r)[-32:]]))
        rest = np.setdiff1d(np.arange(len(s)), i)
        i = np.sort(np.concatenate([i, rng.choice(rest, 64 - len(i), replace=False)])).astype(np.int16)
        idx.append(i), rel.append(a[i]), av.append(b[i])
    samples.update(norm_wise_idx=np.array(idx), norm_wise_release=np.array(rel), norm_wise_avx=np.array(av))

    seed, fs, rate, tw, center, n, n_blocks = t.AVX_RENORM
    taps = po.lpf_design(1.0, fs, rate // 2, tw)
    avx = po.RefFilter(fs // rate, taps, center, fs, n, "avx")
    idx, av = [], []
    for x in t.cu8_blocks(seed, n, n_blocks):
        a = avx.process_cf32("cu8", x, "optimized")
        i = np.sort(rng.choice(len(a), 16, replace=False)).astype(np.int16)  # a seeded 16 of every block
        idx.append(i), av.append(a[i])
    samples.update(avx_optimized_idx=np.array(idx), avx_optimized=np.array(av))

    with open(os.path.join(HERE, "reference_outputs.json"), "w") as f:
        json.dump(out, f, indent=0)
        f.write("\n")
    np.savez_compressed(os.path.join(HERE, "reference_outputs.npz"), **samples)
    print("wrote tests/golden/reference_outputs.json and .npz")


if __name__ == "__main__":
    sys.exit(main())
