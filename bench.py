#!/usr/bin/env python3
"""bench.py -- throughput of the xlating FIR decimator hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--workload cfg2|cfg1|cfg3|c512|c1000|cfg5|cfg5shard] [--taps default|297|2429]
                    [--dump-outputs DIR]

A "step" is ONE REFERENCE QUEUE DEPTH of the wideband stream: 64 blocks
(queue_size, src/config.c:183) of 262144 bytes (buffer_size, src/config.c:208), each
block converted once and NCO-mixed + FIR-filtered + decimated for ALL clients by one
fused launch.  20 steps therefore time ~90 ms of GPU work, not 1.4 ms.
Default workload = BASELINE.json configs[1]: 256 clients on one shared 2.016 Msps cu8
stream, mixed 48/96 ksps, taps from the server's own designer (src/dsp_worker.c:98 with
lpf_cutoff_rate=5 -> 505 / 253 taps).

The JSON line (rank 0):
  value        input MS/s, whole job (each GPU decimates its own independent stream: weak
               scaling, no data-path collective), inputs resident in HBM, outputs left in
               HBM, timed on the device with CUDA events, max over ranks
  e2e          same metric through the batch C ABI with HOST buffers: pinned H2D of every
               block and D2H of every client's output inside the timed region
  e2e_dropin   same workload through the reference's UNMODIFIED per-filter plugin ABI
               (process_*), one dsp thread per client on private copies of every block
  verified     the LAST TIMED block's outputs of 8 sampled clients were copied back and
               compared with the oracle (which replayed the whole block sequence)
  roofline     the dominant kernel against the HBM roofline the metric names (traffic =
               DRAM bytes per launch from an ncu capture taken by this run), plus "fp32":
               the FP32-FMA roofline that actually binds
  cpu_baseline the reference's own CPU path (oracle/_ref/ref_cpu_bench_*: the unmodified
               reference sources, pinned thread-per-client in C) on this box's host cores
  legs         (N > 1) BASELINE configs[3] (c512: 512 clients per GPU) and configs[4]
               (cfg5: ONE 61.44 Msps stream NCCL-broadcast, 4096 clients sharded c mod N)

--impl reference prints the CPU arm alone (same metric/config, a step = 64 blocks).
"""
import argparse
import importlib
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

BLOCK_BYTES = 262144  # src/config.c:208
STEP_BLOCKS = 64      # src/config.c:183 (queue_size): one step = one reference queue depth
N_DEV_BLOCKS = 512    # distinct input blocks rotating through HBM (134 MB > L2)
VERIFY_MAX_BLOCKS = 8192  # longest block history the verification oracle replays


# ---------------------------------------------------------------------------
# workloads (SURVEY.md section 8d)
# ---------------------------------------------------------------------------
def workload(name, taps_mode):
    if name == "cfg2":
        fs, fmt, rates = 2016000, "cu8", [48000 if c % 2 == 0 else 96000 for c in range(256)]
        desc = "cfg2: 256 clients, shared 2.016 Msps cu8 input, mixed 48/96 ksps"
    elif name == "cfg1":
        fs, fmt, rates = 2016000, "cu8", [48000]
        desc = "cfg1: 1 client, 2.016 Msps cu8 -> 48 ksps (perf_xlating shape)"
    elif name == "cfg3":
        fs, fmt, rates = 10000000, "cs16", [250000] * 64
        desc = "cfg3: 64 clients, 10 Msps cs16 -> 250 ksps"
    elif name == "c512":
        fs, fmt, rates = 2016000, "cu8", [48000] * 512
        desc = "cfg4 per-GPU shape: 512 clients, 2.016 Msps cu8 -> 48 ksps"
    elif name == "cfg5":
        # BASELINE configs[4]: ONE 61.44 Msps wideband input, NCCL-broadcast to all GPUs,
        # 4096 clients at 48 ksps sharded over the GPUs (client c -> rank c mod N)
        fs, fmt, rates = 61440000, "cs16", [48000] * 4096
        desc = "cfg5: single 61.44 Msps cs16 input NCCL-broadcast, 4096 clients at 48 ksps sharded c mod N"
    elif name == "cfg5shard":
        fs, fmt, rates = 61440000, "cs16", [48000] * 512
        desc = "cfg5 per-GPU shard: 512 of 4096 clients, 61.44 Msps cs16 -> 48 ksps (15419 taps)"
    elif name == "c1000":
        fs, fmt, rates = 2016000, "cu8", [48000] * 1000
        desc = "target row: 1000 clients, 2.016 Msps cu8 -> 48 ksps"
    else:
        raise SystemExit(f"unknown workload {name}")
    tw_for = {}
    for r in set(rates):
        if taps_mode == "297" and fs == 2016000:
            tw_for[r] = 16400      # -> 297 taps (BASELINE.json's figure, SURVEY.md 0.1)
        elif taps_mode == "297" and fs == 10000000:
            tw_for[r] = 20060      # -> 1201 taps
        elif name == "cfg1" and taps_mode == "2429":
            tw_for[r] = 2000       # test/perf_xlating.c:21
        else:
            tw_for[r] = r // 5     # src/dsp_worker.c:98, lpf_cutoff_rate=5
    C_ = len(rates)
    plan = []
    for c, r in enumerate(rates):
        center = int(round(-fs / 2 + r / 2 + c * (fs - r) / (C_ - 1))) if C_ > 1 else -312000
        plan.append({"rate": r, "decimation": fs // r, "center": center, "cutoff": r // 2, "tw": tw_for[r]})
    elem = 2 if fmt == "cs16" else 1
    return {"name": name, "desc": desc, "fs": fs, "fmt": fmt, "plan": plan,
            "block_elems": BLOCK_BYTES // elem, "block_samples": BLOCK_BYTES // elem // 2}


def workload_config(wl):
    """The `config` object: names the workload and nothing else, identical in both arms."""
    return {"workload": wl["desc"], "clients": len(wl["plan"]), "fs": wl["fs"], "input": wl["fmt"],
            "block_bytes": BLOCK_BYTES, "blocks_per_step": STEP_BLOCKS,
            "taps": sorted({(p["rate"], p["tw"]) for p in wl["plan"]}),
            "streams": "one independent stream per GPU",
            "l2": f"inputs larger than L2 ({N_DEV_BLOCKS} distinct blocks = {N_DEV_BLOCKS * BLOCK_BYTES // 1000000} MB)"}


def synth_blocks(fmt, n_blocks, block_elems, seed):
    rng = np.random.default_rng(seed)
    if fmt == "cu8":
        return rng.integers(0, 256, (n_blocks, block_elems), dtype=np.uint8)
    if fmt == "cs8":
        return rng.integers(-128, 128, (n_blocks, block_elems), dtype=np.int8)
    return rng.integers(-8192, 8192, (n_blocks, block_elems), dtype=np.int16)


# ---------------------------------------------------------------------------
# clocks sampler (B200_PROFILING.md "clocks DURING the timed region")
# ---------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,power.draw")

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.gpu = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), line.strip()))

    def mark(self):
        return time.perf_counter()

    def stop(self, window=None):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, sm_timed, mx, reasons, power = [], [], None, set(), []
        for ts, r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 6:
                continue
            try:
                v = float(f[0])
                mx = float(f[1])
            except ValueError:
                continue
            sm.append(v)
            if window and window[0] <= ts <= window[1]:
                sm_timed.append(v)
            try:
                power.append(float(f[6]))
            except (ValueError, IndexError):
                pass
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[2:6]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        load = sm_timed if sm_timed else (sm[len(sm) // 2:] if sm else [])
        return {"sm_mhz": float(np.median(load)) if load else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm), "samples_in_timed_region": len(sm_timed),
                "power_w_max": max(power) if power else None}


# ---------------------------------------------------------------------------
# CPU arm: the reference's own implementation, pinned thread-per-client in C
# (oracle/ref_cpu_bench.c + the unmodified reference sources; src/dsp_worker.c:41-88 model)
# ---------------------------------------------------------------------------
def cpu_flags():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("flags"):
                return set(line.split(":", 1)[1].split())
    except OSError:
        pass
    return set()


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except OSError:
        pass
    return "unknown"


CPU_VARIANTS = [  # (binary suffix, gcc flags on top of -O3 -DNDEBUG -ffast-math, cpu flags it needs)
    ("release", "(what CMake Release ships: no -m flags, SIMD not detected)", set()),
    ("avx", "-mavx2 -mfma", {"avx2", "fma"}),
    ("v3", "-march=x86-64-v3", {"avx2", "fma", "bmi2"}),
    ("v4", "-march=x86-64-v4 (stand-in for -march=native on AVX-512 hosts)", {"avx512f", "avx512bw", "avx512vl", "avx512dq"}),
]


CPU_MODES = [  # (label, extra argv after <native|optimized>): max_threads, pin|nopin, main|local
    ("pinned, one thread per logical CPU, filters created by the main thread (the reference's acceptor-thread model)",
     ["0", "pin", "main"]),
    ("unpinned, one thread per logical CPU, filters created by the main thread", ["0", "nopin", "main"]),
    ("pinned, one thread per logical CPU, each thread creates its own filters (NUMA-local working buffers)",
     ["0", "pin", "local"]),
    ("pinned, one thread per PHYSICAL core, each thread creates its own filters", ["half", "pin", "local"]),
]


def cpu_arm(wl, blocks, warmup_blocks, variants=("avx", "v3", "v4", "release"), seconds_cap=60.0):
    """Runs oracle/_ref/ref_cpu_bench_<variant> (the reference compiled from its own sources;
    pinned thread-per-client in C, BASELINE.md section 3).  The threading mode is chosen by a
    short probe of four modes with the AVX build, then every flag set this CPU supports is
    timed in that mode and the FASTEST is quoted, so that the comparison is not flattering."""
    ref_dir = os.path.join(ROOT, "oracle", "_ref")
    flags = cpu_flags()
    plan = "\n".join(f"{p['decimation']} {p['cutoff']} {p['tw']} {p['center']}" for p in wl["plan"]) + "\n"
    ncpu = len(os.sched_getaffinity(0))

    def run(name, nblocks, nwarm, mode):
        exe = os.path.join(ref_dir, f"ref_cpu_bench_{name}")
        extra = [str(max(1, ncpu // 2)) if a == "half" else a for a in mode]
        r = subprocess.run([exe, str(wl["fs"]), wl["fmt"], str(wl["block_elems"]), str(nblocks), str(nwarm),
                            "optimized"] + extra, input=plan, capture_output=True, text=True, timeout=600)
        return json.loads(r.stdout.strip().splitlines()[-1])

    t_start = time.perf_counter()
    probe_exe = next((n for n in ("avx", "release") if os.path.exists(os.path.join(ref_dir, f"ref_cpu_bench_{n}"))
                      and (n == "release" or {"avx2", "fma"} <= flags)), None)
    if probe_exe is None:
        raise RuntimeError("oracle/_ref/ref_cpu_bench_* not built (oracle/_ref is built where /root/reference exists)")
    probes = {}
    for label, mode in CPU_MODES:
        try:
            probes[label] = run(probe_exe, 48, 8, mode)["input_msps"]
        except Exception as ex:  # noqa: BLE001
            probes[label] = repr(ex)
    good = {k: v for k, v in probes.items() if isinstance(v, float)}
    if not good:
        raise RuntimeError(f"no reference CPU run succeeded: {probes}")
    best_label = max(good, key=good.get)
    best_mode = dict(CPU_MODES)[best_label]
    runs = {}
    for name, gcc, need in CPU_VARIANTS:
        if name not in variants:
            continue
        if not os.path.exists(os.path.join(ref_dir, f"ref_cpu_bench_{name}")):
            runs[name] = {"skipped": "not built"}
        elif not need <= flags:
            runs[name] = {"skipped": f"this CPU lacks {sorted(need - flags)}"}
        elif runs and time.perf_counter() - t_start > seconds_cap:
            runs[name] = {"skipped": "time budget of the CPU leg spent"}
        else:
            try:
                d = run(name, blocks, warmup_blocks, best_mode)
                d["gcc_flags"] = "-O3 -DNDEBUG -ffast-math " + gcc
                runs[name] = d
            except Exception as ex:  # noqa: BLE001
                runs[name] = {"error": repr(ex)}
    ok = {k: v for k, v in runs.items() if "input_msps" in v}
    if not ok:
        raise RuntimeError(f"no reference CPU binary could run: {runs}")
    best = max(ok, key=lambda k: ok[k]["input_msps"])
    b = ok[best]
    return {"value": b["input_msps"], "unit": "MS/s", "cores": b["threads"], "kind": "reference",
            "sample": f"{b['blocks']} blocks of {BLOCK_BYTES} B through all {b['clients']} clients after "
                      f"{b['warmup_blocks']} warm-up blocks; {b['threads']} threads: {best_label}; thread-per-client "
                      f"(src/dsp_worker.c:41-88 without I/O and queue memcpy); oracle/_ref/ref_cpu_bench_{best} = "
                      f"unmodified reference sources, gcc {b['gcc_flags']}, process_optimized_* "
                      f"(SIMD_STATUS={b['simd_status']}), wall {b['seconds']:.2f} s",
            "client_msps": b["client_msps"], "best_variant": best, "cpu_model": cpu_model(), "nproc": os.cpu_count(),
            "threading_probe_msps": {k: (round(v, 3) if isinstance(v, float) else v) for k, v in probes.items()},
            "variants": {k: (round(v["input_msps"], 3) if "input_msps" in v else v) for k, v in runs.items()}}


# ---------------------------------------------------------------------------
# multi-GPU plumbing (one process per GPU; the only collectives on the default path are
# the barrier and the max-over-ranks of the timed region)
# ---------------------------------------------------------------------------
def stream_seed(rank):
    """Each rank decimates its OWN wideband stream (weak scaling, SURVEY 8e)."""
    return 1000 + rank


def max_over_ranks(x, world, device=None):
    """MAX all-reduce of a python float (NCCL on GPU boxes, gloo in the CPU tests)."""
    if world <= 1:
        return float(x)
    import torch
    import torch.distributed as dist
    t = torch.tensor([x], dtype=torch.float64, device=device if device is not None else "cpu")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def min_over_ranks(x, world, device=None):
    return -max_over_ranks(-float(x), world, device)


def job_throughput_msps(block_samples, blocks, world, elapsed_ms_max):
    """Whole-job input MS/s: every rank pushed `blocks` blocks of its own stream."""
    return world * block_samples * blocks / (elapsed_ms_max * 1e-3) / 1e6


def shard_clients(n_clients, rank, world):
    """configs[4] partitioning: client c belongs to rank c mod world."""
    return list(range(rank, n_clients, world))


ORIG_AFFINITY = None  # set by numa_bind; numa_unbind restores it for the CPU legs (they use every core)


def numa_unbind():
    if ORIG_AFFINITY is not None:
        os.sched_setaffinity(0, ORIG_AFFINITY)


def numa_bind(local_rank):
    """Bind this rank (and therefore its pinned allocations, first-touch) to the CPUs of its
    GPU's NUMA node: eight ranks writing D2H results into one node's DRAM was what bent the
    round-1 end-to-end scaling curve (VERDICT item 6).  Returns a description or None."""
    try:
        out = subprocess.run(["nvidia-smi", "topo", "-m"], capture_output=True, text=True, timeout=20).stdout
        for line in out.splitlines():
            cols = line.split("\t")
            if cols and cols[0].strip().replace("\x1b[4m", "") == f"GPU{local_rank}":
                for c in cols:
                    c = c.strip()
                    if c and all(ch.isdigit() or ch in ",-" for ch in c) and ("-" in c or "," in c):
                        cpus = set()
                        for part in c.split(","):
                            a, _, b = part.partition("-")
                            cpus |= set(range(int(a), int(b or a) + 1))
                        cpus &= os.sched_getaffinity(0)
                        if cpus:
                            global ORIG_AFFINITY
                            if ORIG_AFFINITY is None:
                                ORIG_AFFINITY = os.sched_getaffinity(0)
                            os.sched_setaffinity(0, cpus)
                            return f"rank bound to CPUs {c} (GPU{local_rank}'s NUMA node)"
    except Exception:  # noqa: BLE001
        pass
    return None


# ---------------------------------------------------------------------------
# verification against the oracle (checker only)
# ---------------------------------------------------------------------------
def verify_last_block(pkg, g, wl, ids, tapsets, block_seq, get_block, ticket, sample, read):
    """Compare the outputs of `ticket` (the last block of block_seq) for the sampled clients
    with the oracle, which replays the whole block sequence (history + oscillator state)."""
    from concurrent.futures import ThreadPoolExecutor

    from oracle import pyoracle as po  # checker only

    def one(c):
        p = wl["plan"][c]
        o = po.OracleFilter(p["decimation"], tapsets[(p["cutoff"], p["tw"])], p["center"], wl["fs"], wl["block_elems"])
        y = None
        for b in block_seq:
            y = o.process_cf32(wl["fmt"], get_block(b))
        got = read(ticket, ids[c])
        if got.shape != y.shape:
            return float("inf")
        scale = float(np.max(np.abs(y)))
        d = np.abs(got.astype(np.complex128) - y.astype(np.complex128))
        norm = float(d.max() / scale)
        elem_ok = bool(np.all(d <= 1e-5 * np.abs(y) + 1e-5 * scale))
        return norm if elem_ok else max(norm, 1.0)

    with ThreadPoolExecutor(max_workers=len(sample)) as ex:
        errs = list(ex.map(one, sample))
    worst = max(errs)
    return {"ok": bool(worst <= 1e-5), "max_normwise_error": worst, "tolerance": 1e-5, "clients_checked": list(sample),
            "blocks_replayed_by_oracle": len(block_seq),
            "what": "last timed block, outputs copied back from HBM, oracle/liboracle.so replayed every block "
                    "since the group was created"}


DUMP_BYTES = 64 << 20  # --dump-outputs budget


def dump_outputs(pkg, g, ids, last, out_dir):
    """--dump-outputs: what the timed path handed its callers for the last blocks of the
    last timed step, written as out_dir/client_<c>.npy (float32 [n, 2] = re, im): client c's
    outputs of those blocks, concatenated.  The blocks are the XLG_SLOTS whose device output
    arenas are still live after the final wait; clients are taken in a fixed seeded order
    while their outputs fit DUMP_BYTES."""
    os.makedirs(out_dir, exist_ok=True)
    tickets = range(last - pkg.XLG_SLOTS + 1, last + 1)
    total = 0
    for c in np.random.default_rng(0).permutation(len(ids)):
        nbytes = 8 * sum(g.output_ptr(t, ids[c])[1] for t in tickets)
        if total + nbytes > DUMP_BYTES:
            continue
        y = np.concatenate([g.read_output(t, ids[c]) for t in tickets])
        np.save(os.path.join(out_dir, f"client_{c:04d}.npy"), y.view(np.float32).reshape(-1, 2))
        total += nbytes


# ---------------------------------------------------------------------------
# DRAM traffic of the dominant kernel: one ncu capture taken by THIS run
# ---------------------------------------------------------------------------
def run_probe(args):
    """--probe: push a few blocks through the value-leg configuration and exit (run under
    ncu by measure_traffic; no torch, no timing)."""
    pkg = importlib.import_module("sdr-server_b200")
    wl = workload(args.workload, args.taps)
    g = pkg.Group(wl["fs"], wl["block_elems"], flags=pkg.XLG_OUT_DEVICE)
    tapsets = {}
    for p in wl["plan"]:
        key = (p["cutoff"], p["tw"])
        if key not in tapsets:
            tapsets[key] = pkg.create_low_pass_filter(1.0, wl["fs"], p["cutoff"], p["tw"])
        g.add_client(p["decimation"], tapsets[key], p["center"])
    blocks = synth_blocks(wl["fmt"], 8, wl["block_elems"], seed=7)
    last = -1
    for i in range(16):
        last = g.submit(wl["fmt"], blocks[i % 8])
    g.wait(last)
    g.close()
    return 0


def measure_traffic(args, kernel_regex):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from an
    `ncu` capture of `bench.py --probe` taken now (never of the timed run itself)."""
    tmp = tempfile.NamedTemporaryFile(prefix="xl_traffic_", suffix=".csv", delete=False)
    tmp.close()
    cmd = ["ncu", "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum", "--clock-control", "none",
           "--print-units", "base", "-k", f"regex:{kernel_regex}", "-s", "6", "-c", "6", "--csv", "--log-file", tmp.name,
           sys.executable, os.path.abspath(__file__), "--probe", "--workload", args.workload, "--taps", args.taps]
    try:
        subprocess.run(cmd, capture_output=True, text=True, timeout=240, check=True)
        import csv
        rd, wr = [], []
        with open(tmp.name) as f:
            rows = [r for r in csv.reader(f) if len(r) > 3]
        hdr = next(r for r in rows if "Metric Name" in r)
        mi, vi = hdr.index("Metric Name"), hdr.index("Metric Value")
        for r in rows:
            if r is hdr or len(r) <= vi:
                continue
            if r[mi] == "dram__bytes_read.sum":
                rd.append(float(r[vi].replace(",", "")))
            elif r[mi] == "dram__bytes_write.sum":
                wr.append(float(r[vi].replace(",", "")))
        if not rd:
            raise RuntimeError("no matching launches in the ncu log")
        return {"traffic": float(np.mean(rd) + np.mean(wr)), "read": float(np.mean(rd)), "write": float(np.mean(wr)),
                "launches": len(rd), "source": "ncu capture taken by this run (bench.py --probe under ncu --metrics "
                                               "dram__bytes_read.sum,dram__bytes_write.sum --clock-control none)"}
    except Exception as ex:  # noqa: BLE001
        return {"traffic": None, "source": f"ncu capture failed: {ex!r}"[:300]}
    finally:
        try:
            os.unlink(tmp.name)
        except OSError:
            pass


# ---------------------------------------------------------------------------
# the standard leg: one independent stream on this rank's GPU
# ---------------------------------------------------------------------------
def run_stream_leg(pkg, wl, args, rank, world, local_rank, steps, warmup, partition=True, full=True):
    """value (device-timed, inputs and outputs in HBM), verification of the last timed block,
    block latency, per-kernel profile and e2e (host buffers) for one workload.  `full`
    adds the latency / profile passes (headline leg only)."""
    import torch
    import torch.distributed as dist

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    tapsets = {}

    def build_group(flags):
        g = pkg.Group(wl["fs"], wl["block_elems"], device=local_rank, flags=flags)
        ids = []
        for p in wl["plan"]:
            key = (p["cutoff"], p["tw"])
            if key not in tapsets:
                tapsets[key] = pkg.create_low_pass_filter(1.0, wl["fs"], p["cutoff"], p["tw"])
            ids.append(g.add_client(p["decimation"], tapsets[key], p["center"]))
        return g, ids

    fmt_code = pkg.FMT[wl["fmt"]]
    host_blocks = synth_blocks(wl["fmt"], N_DEV_BLOCKS, wl["block_elems"], seed=stream_seed(rank))
    dev = torch.from_numpy(host_blocks.view(np.uint8).reshape(N_DEV_BLOCKS, -1)).cuda()
    blk_stride, base_ptr = dev.stride(0), dev.data_ptr()

    # ---- tier (i): inputs resident in HBM, outputs stay in HBM -> `value`
    part_flag = pkg.XLG_SM_PARTITION if partition else 0
    g, ids = build_group(pkg.XLG_OUT_DEVICE | part_flag)
    seq = []  # every block index submitted to g, in order (the oracle replays it)

    def run_blocks(k):
        last = -1
        for _ in range(k):
            b = len(seq) % N_DEV_BLOCKS
            seq.append(b)
            last = g.submit_ptr(fmt_code, base_ptr + b * blk_stride, wl["block_elems"], pkg.XLG_INPUT_DEVICE)
        return last

    g.wait(run_blocks(warmup * STEP_BLOCKS))
    g.profile_read(reset=True)
    barrier()
    t_wall0 = time.perf_counter()
    g.timer_start()
    last = run_blocks(steps * STEP_BLOCKS)
    ms = g.timer_stop()
    t_wall1 = time.perf_counter()
    host = g.profile_read(reset=True)
    barrier()
    g.wait(last)
    if full and rank == 0 and args.dump_outputs:
        dump_outputs(pkg, g, ids, last, args.dump_outputs)
    n_out_total = sum(g.output_ptr(last, c)[1] for c in ids)
    out = {"timed_window": (t_wall0, t_wall1), "n_out_total": n_out_total, "tapsets": tapsets,
           "partition_sms": g.partition_sms()}

    # ---- the last TIMED block, every sampled client, against the oracle
    if args.no_verify:
        out["verified"] = {"ok": None, "what": "skipped (--no-verify)"}
    elif len(seq) <= VERIFY_MAX_BLOCKS:
        C_ = len(ids)
        sample = sorted({0, 1, C_ // 4, C_ // 4 + 1, C_ // 2, C_ // 2 + 1, C_ - 2, C_ - 1} & set(range(C_)))
        out["verified"] = verify_last_block(pkg, g, wl, ids, tapsets, list(seq), lambda b: host_blocks[b], last, sample,
                                            g.read_output)
    else:
        out["verified"] = {"ok": None, "what": f"skipped: {len(seq)} blocks of history exceed the "
                                               f"{VERIFY_MAX_BLOCKS}-block budget of the replaying oracle"}

    if full:
        # latency pass: one block at a time (submit, wait), as a real-time server sees it
        lat = []
        for _ in range(100):
            t0 = time.perf_counter()
            g.wait(run_blocks(1))
            lat.append(time.perf_counter() - t0)
        out["block_latency_us"] = {"median": float(np.median(lat)) * 1e6, "p95": float(np.percentile(lat, 95)) * 1e6,
                                   "what": "host wall clock submit->wait of ONE block, input and outputs in HBM, "
                                           "pipeline otherwise idle"}
        # per-kernel pass (CUDA events around every launch, on the launching stream)
        g.profile_enable(True)
        g.profile_read(reset=True)
        g.wait(run_blocks(256))
        g.profile_enable(False)
        out["prof"] = g.profile_read(reset=True)
    out["kinds"] = sorted({g.client_info(c)[1] for c in ids})
    out["host"] = {"submit_us_per_block": 1e3 * host["host_submit_ms"] / max(host["submits"], 1),
                   "of_which_waiting_for_gpu_us": 1e3 * host["host_wait_ms"] / max(host["submits"], 1)}
    g.close()
    out["ms_max"] = max_over_ranks(ms, world, "cuda")
    out["blocks"] = steps * STEP_BLOCKS
    out["value"] = job_throughput_msps(wl["block_samples"], out["blocks"], world, out["ms_max"])

    # ---- tier (iii): through the batch C ABI with host buffers -> `e2e`
    if not args.no_e2e:
        g2, ids2 = build_group(0)
        n_pin = 8
        pins = [pkg.PinnedBuffer(BLOCK_BYTES) for _ in range(n_pin)]
        for i, p in enumerate(pins):
            p.array(np.uint8)[:] = host_blocks[i].view(np.uint8)
        sink = [0.0]
        import ctypes as C

        def consume(tk):
            # the results are in pinned host memory: read one float of every 16 KiB of this
            # block's output arena (all clients), like consumers that would now write them out
            p0, _ = g2.output_ptr(tk, ids2[0])
            p1, n1 = g2.output_ptr(tk, ids2[-1])
            nfl = (p1 - p0) // 4 + 2 * n1
            arr = np.ctypeslib.as_array(C.cast(p0, C.POINTER(C.c_float)), shape=(nfl,))
            sink[0] += float(arr[::4096].sum())

        def run_e2e(k):
            pend = []
            for s in range(k):
                pend.append(g2.submit_ptr(fmt_code, pins[s % n_pin].ptr, wl["block_elems"], pkg.XLG_INPUT_KEEP))  # 8 rotating pinned blocks
                if len(pend) >= pkg.XLG_SLOTS - 1:
                    tk = pend.pop(0)
                    g2.wait(tk)
                    consume(tk)
            for tk in pend:
                g2.wait(tk)
                consume(tk)

        run_e2e(warmup * STEP_BLOCKS)
        barrier()
        t0 = time.perf_counter()
        run_e2e(steps * STEP_BLOCKS)
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        barrier()
        wall = max_over_ranks(wall, world, "cuda")
        out["e2e"] = {"value": job_throughput_msps(wl["block_samples"], steps * STEP_BLOCKS, world, wall * 1e3),
                      "unit": "MS/s", "h2d_bytes_per_step": BLOCK_BYTES * STEP_BLOCKS,
                      "d2h_bytes_per_step": int(n_out_total * 8) * STEP_BLOCKS, "steps": steps,
                      "ms_per_step": wall * 1e3 / steps,
                      "timing": "host wall clock around submit..wait of every block, max over ranks; pinned host input "
                                "blocks, every client's output copied to pinned host memory and read by the host"}
        g2.close()
        for p in pins:
            p.free()
        # what bounds e2e: the D2H copy of every client's output.  Measure the copy engine's own ceiling on
        # this box (pinned host buffer, same size as one step's results) and report the link's share.
        try:
            nbytes = int(min(max(n_out_total * 8 * STEP_BLOCKS, 64 << 20), 512 << 20))
            d_buf = torch.empty(nbytes, dtype=torch.uint8, device="cuda")
            h_buf = torch.empty(nbytes, dtype=torch.uint8).pin_memory()
            ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            best = 1e30
            for _ in range(4):
                ev0.record()
                h_buf.copy_(d_buf, non_blocking=True)
                ev1.record()
                ev1.synchronize()
                best = min(best, ev0.elapsed_time(ev1))
            peak = nbytes / (best * 1e-3) / 1e9
            used = out["e2e"]["d2h_bytes_per_step"] / (out["e2e"]["ms_per_step"] * 1e-3) / 1e9
            out["e2e"]["pcie"] = {"d2h_gbs": used, "d2h_peak_gbs": peak, "frac": used / peak,
                                  "what": "bytes of results copied to the host per second of e2e wall clock, against a "
                                          "plain pinned cudaMemcpy D2H of the same size measured in this run"}
            del d_buf, h_buf
        except Exception as e:  # noqa: BLE001
            out["e2e"]["pcie"] = {"error": str(e)}
    return out


# ---------------------------------------------------------------------------
# BASELINE configs[4]: one wideband stream, NCCL-broadcast, clients sharded
# ---------------------------------------------------------------------------
def run_broadcast_leg(pkg, wl, args, rank, world, local_rank, steps, warmup):
    """Rank 0 owns the stream (synthetic blocks in its HBM, or in pinned host memory for e2e)
    and NCCL-broadcasts each block; every rank decimates its own shard of the clients from
    the received buffer (xlg_wait_stream + XLG_INPUT_DEVICE: the kernel consumes the NCCL
    receive buffer directly, no staging copy).  Strong scaling: the job's work is fixed,
    `value` is the input rate of the ONE stream."""
    import torch
    import torch.distributed as dist

    dev = torch.device("cuda", local_rank)
    mine = shard_clients(len(wl["plan"]), rank, world)
    plan = [wl["plan"][c] for c in mine]
    fmt_code = pkg.FMT[wl["fmt"]]
    taps = pkg.create_low_pass_filter(1.0, wl["fs"], plan[0]["cutoff"], plan[0]["tw"])

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def make_group(flags):
        g = pkg.Group(wl["fs"], wl["block_elems"], device=local_rank, flags=flags)
        return g, [g.add_client(p["decimation"], taps, p["center"]) for p in plan]

    n_src = 64
    src_host = synth_blocks(wl["fmt"], n_src, wl["block_elems"], seed=stream_seed(0))  # same on every rank (checker)
    nbytes = src_host[0].nbytes
    src_dev = torch.from_numpy(src_host.view(np.uint8).reshape(n_src, -1)).to(dev) if rank == 0 else None
    pinned = torch.from_numpy(src_host.view(np.uint8).reshape(n_src, -1)).pin_memory() if rank == 0 else None
    ring = [torch.empty(nbytes, dtype=torch.uint8, device=dev) for _ in range(pkg.XLG_SLOTS)]
    stream = torch.cuda.current_stream()
    seq = []

    def pump(g, blocks, from_host, record=None):
        """broadcast + submit `blocks` blocks, keeping at most XLG_SLOTS-1 tickets in flight"""
        pend, last = [], -1
        for i in range(blocks):
            buf = ring[i % len(ring)]
            if len(pend) >= len(ring) - 1:
                g.wait(pend.pop(0))  # the block that used this buffer has been converted
            if rank == 0:
                buf.copy_(pinned[i % n_src] if from_host else src_dev[i % n_src], non_blocking=True)
            if world > 1:
                dist.broadcast(buf, src=0)
            g.wait_stream(stream.cuda_stream)
            last = g.submit_ptr(fmt_code, buf.data_ptr(), wl["block_elems"], pkg.XLG_INPUT_DEVICE)
            pend.append(last)
            if record is not None:
                record.append(i % n_src)
        for t in pend:
            g.wait(t)
        return last

    g, ids = make_group(pkg.XLG_OUT_DEVICE)
    pump(g, warmup * STEP_BLOCKS, False, seq)
    barrier()
    g.timer_start()
    last = pump(g, steps * STEP_BLOCKS, False, seq)
    ms = g.timer_stop()
    barrier()
    if rank == 0 and args.dump_outputs:
        dump_outputs(pkg, g, ids, last, args.dump_outputs)
    ms_max = max_over_ranks(ms, world, "cuda")
    # every rank checks 4 of ITS clients of the last timed block against the oracle
    ok, worst = 1.0, 0.0
    if not args.no_verify and len(seq) <= VERIFY_MAX_BLOCKS:
        sample = sorted({0, len(ids) // 3, 2 * len(ids) // 3, len(ids) - 1})
        shard_wl = dict(wl, plan=plan)
        v = verify_last_block(pkg, g, shard_wl, ids, {(plan[0]["cutoff"], plan[0]["tw"]): taps}, list(seq),
                              lambda b: src_host[b], last, sample, g.read_output)
        ok, worst = (1.0 if v["ok"] else 0.0), v["max_normwise_error"]
    ok = min_over_ranks(ok, world, "cuda")
    worst = max_over_ranks(worst, world, "cuda")
    g.profile_enable(True)
    g.profile_read(reset=True)
    pump(g, 32, False)
    g.profile_enable(False)
    prof = g.profile_read(reset=True)
    kinds = sorted({g.client_info(c)[1] for c in ids})
    g.close()
    value = wl["block_samples"] * steps * STEP_BLOCKS / (ms_max * 1e-3) / 1e6  # ONE stream

    g2, _ = make_group(0)
    pump(g2, warmup * STEP_BLOCKS, True)
    barrier()
    t0 = time.perf_counter()
    pump(g2, steps * STEP_BLOCKS, True)
    torch.cuda.synchronize()
    wall = max_over_ranks(time.perf_counter() - t0, world, "cuda")
    barrier()
    g2.close()
    n_out_per_block = len(wl["plan"]) * (wl["block_samples"] // plan[0]["decimation"])
    k_ms = (prof["fir_long_ms"] / max(prof["fir_long_launches"], 1)) or (prof["fir_tile_ms"] / max(prof["fir_tile_launches"], 1))
    algo_fma = 4.0 * prof["algo_macs"] / max(prof["blocks"], 1)
    return {"workload": wl["desc"], "scaling": "strong", "value": value, "unit": "MS/s",
            "ms_per_step": ms_max / steps, "steps": steps, "blocks_per_step": STEP_BLOCKS,
            "realtime_factor": value * 1e6 / wl["fs"], "clients_per_gpu": len(plan), "taps_len": len(taps),
            "kernels_used": kinds,
            "parallelism": f"clients sharded c mod {world}; every block NCCL-broadcast from rank 0 into a ring of "
                           f"{pkg.XLG_SLOTS} receive buffers the FIR reads directly",
            "verified": {"ok": bool(ok >= 1.0), "max_normwise_error": worst,
                         "what": "last timed block, 4 clients per rank, oracle replayed the whole block sequence"},
            "e2e": {"value": wl["block_samples"] * steps * STEP_BLOCKS / wall / 1e6, "unit": "MS/s",
                    "h2d_bytes_per_step": nbytes * STEP_BLOCKS, "d2h_bytes_per_step": int(n_out_per_block * 8) * STEP_BLOCKS,
                    "timing": "host wall clock, max over ranks; rank 0 copies each block from pinned host memory, NCCL "
                              "broadcast, every rank copies its clients' outputs back to pinned host memory"},
            "fir_kernel_ms_per_rank": k_ms,
            "fp32_frac_kernel": algo_fma / (k_ms * 1e-3) / 1e12 / 36.2 if k_ms else None}


def dropin_leg(wl, blocks=48, window=64):
    """The same workload through the reference's UNMODIFIED per-filter ABI and threading
    model (one filter + one dsp thread per client, private copies of every block,
    src/dsp_worker.c:41-88 / src/queue.c:114): what sdr-server gets by re-linking only."""
    exe = os.path.join(ROOT, "sdr-server_b200", "bin", "dropin_bench")
    out = subprocess.run([exe, str(len(wl["plan"])), str(blocks), str(window)], capture_output=True, text=True,
                         timeout=300).stdout
    d = json.loads(out.strip().splitlines()[-1])
    return {"value": d["input_msps"], "unit": "MS/s", "clients": d["clients"], "threads": d["clients"],
            "blocks": d["blocks"], "queue_window": d["window"], "calls_per_s": d["calls_per_s"],
            "launch_batches": d["launch_batches"], "shared_inputs": d["shared_inputs"],
            "engine_calls": d["engine_calls"], "stream_blocks": d.get("stream_blocks"),
            "stream_hits": d.get("stream_hits"),
            "h2d_bytes_per_step": None, "d2h_bytes_per_step": None,
            "note": "process_native_cu8_cf32 from one thread per client on private block copies "
                    "(sdr-server_b200/host/dropin_bench.c); host wall clock"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="cfg2")
    ap.add_argument("--taps", default="default")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--no-traffic", action="store_true", help="skip the ncu capture of the dominant kernel's DRAM traffic")
    ap.add_argument("--no-dropin", action="store_true",
                    help="skip the thread-per-client run of the unmodified per-filter ABI (bin/dropin_bench)")
    ap.add_argument("--no-partition", action="store_true",
                    help="do not reserve 8 SMs (green context) for the oscillator pre-pass")
    ap.add_argument("--no-legs", action="store_true", help="N > 1: skip the c512 and cfg5 legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the outputs of the last timed blocks as DIR/client_<c>.npy")
    ap.add_argument("--probe", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.probe:
        return run_probe(args)
    if args.warmup < 3:
        args.warmup = 3

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    wl = workload(args.workload, args.taps)
    config = workload_config(wl)

    # ------------------------------------------------------------------ CPU arm
    if args.impl == "reference":
        if rank != 0:
            return 0
        t0 = time.perf_counter()
        # a step = 64 blocks through all clients; bounded so that the run ends within minutes
        blocks = max(STEP_BLOCKS, min(args.steps * STEP_BLOCKS, 2560))
        r = cpu_arm(wl, blocks=blocks, warmup_blocks=min(args.warmup * STEP_BLOCKS, 64), variants=("avx", "v4"))
        ms_per_step = wl["block_samples"] * STEP_BLOCKS / r["value"] / 1e3
        line = {"metric": "IQ MS/s in", "value": r["value"], "unit": "MS/s", "n_gpus": args.gpus, "steps": args.steps,
                "warmup": args.warmup, "ms_per_step": ms_per_step,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                "data": "synthetic", "impl": "reference", "config": config, "cpu_baseline": r,
                "e2e": {"value": r["value"], "unit": "MS/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                "gpu_launches": 0, "wall_s": time.perf_counter() - t0}
        print(json.dumps(line))
        return 0

    # ------------------------------------------------------------------ GPU arm
    # pinned host buffers are first-touched by this process: keep it (and them) on the GPU's NUMA node --
    # a run that happens to start on the far socket loses a third of its D2H bandwidth (752 -> 527 MS/s e2e)
    numa = numa_bind(local_rank)
    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl b200 needs a CUDA device (no CPU fallback)")
    torch.cuda.set_device(local_rank)
    if world > 1:
        # rank 0 must print exactly ONE line on stdout, but NCCL prints its version banner
        # there when the first communicator is created: point fd 1 at stderr while that happens
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
            warm = torch.zeros(1, device="cuda")
            dist.all_reduce(warm)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    pkg = importlib.import_module("sdr-server_b200")
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()

    if wl["name"] == "cfg5":
        leg = run_broadcast_leg(pkg, wl, args, rank, world, local_rank, args.steps, args.warmup)
        clocks = sampler.stop() if rank == 0 else None
        if rank == 0:
            config["streams"] = "ONE wideband stream for the whole job"
            line = {"metric": "IQ MS/s in", "value": leg["value"], "unit": "MS/s", "n_gpus": world, "steps": args.steps,
                    "warmup": args.warmup, "ms_per_step": leg["ms_per_step"], "higher_is_better": True,
                    "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                    "verified": leg["verified"]["ok"], "verification": leg["verified"], "clocks": clocks,
                    "e2e": leg["e2e"], "gpu_launches": 3 * args.steps * STEP_BLOCKS, "engine": leg}
            print(json.dumps(line))
        if world > 1:
            dist.destroy_process_group()
        return 0

    main_leg = run_stream_leg(pkg, wl, args, rank, world, local_rank, args.steps, args.warmup,
                              partition=not args.no_partition, full=True)
    legs = {}
    if world > 1 and not args.no_legs and args.workload == "cfg2":
        # BASELINE configs[3] and configs[4] on the driver's record (VERDICT item 5); shorter than the headline
        k = max(3, min(args.steps, 10))
        c512 = run_stream_leg(pkg, workload("c512", "default"), args, rank, world, local_rank, k, 3,
                              partition=not args.no_partition, full=False)
        legs["c512"] = {"workload": f"BASELINE configs[3]: {world} independent 2.016 Msps streams x 512 clients "
                                    "(one stream per GPU), 505 taps",
                        "scaling": "weak", "value": c512["value"], "unit": "MS/s",
                        "ms_per_step": c512["ms_max"] / k, "steps": k, "blocks_per_step": STEP_BLOCKS,
                        "e2e": c512.get("e2e"), "verified": c512["verified"], "kernels_used": c512["kinds"]}
        legs["cfg5"] = run_broadcast_leg(pkg, workload("cfg5", "default"), args, rank, world, local_rank, k, 3)

    clocks = sampler.stop(window=main_leg["timed_window"]) if rank == 0 else None
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    # ---- roofline of the dominant kernel
    prof = main_leg["prof"]
    ms_max, blocks = main_leg["ms_max"], main_leg["blocks"]
    ms_per_block = ms_max / blocks
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:  # noqa: BLE001
        pass
    hbm_peak = peaks.get("hbm_gbs", 6650.0)
    peak_src = "MEASURED_PEAKS.json hbm_gbs (burst copy)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s"
    algo_bytes = BLOCK_BYTES + 8 * main_leg["n_out_total"]  # read the block once, write cf32 per client (SURVEY 8d)
    dom = max(("fir_tile", "fir_long", "fir_generic"), key=lambda k: prof[f"{k}_ms"])
    kname = {"fir_tile": "fir_tile_cf32_kernel", "fir_long": "fir_long4_cf32_kernel (XLATING_B200_LONG picks 1-4) + fir_long_reduce_kernel",
             "fir_generic": "fir_generic_cf32_kernel"}[dom]
    kregex = {"fir_tile": "fir_tile_cf32_kernel", "fir_long": "fir_long[0-9]?_cf32_kernel",
              "fir_generic": "fir_generic_cf32_kernel"}[dom]
    roof = {"bound": "hbm", "achieved": None, "peak": hbm_peak, "unit": "GB/s", "frac": None, "traffic": None,
            "peak_source": peak_src, "kernel": kname, "algorithmic_bytes_per_launch": algo_bytes,
            "launch": "one launch = one 262144-byte block through all clients"}
    if world == 1 and not args.no_traffic:
        tr = measure_traffic(args, kregex)
        roof["traffic"] = tr.pop("traffic")
        roof["traffic_detail"] = tr
    else:
        roof["traffic_detail"] = {"source": "not captured (ncu never wraps a multi-rank run)" if world > 1 else "--no-traffic"}
    if prof[f"{dom}_launches"] > 0:
        k_ms = prof[f"{dom}_ms"] / prof[f"{dom}_launches"]
        roof["kernel_ms"] = k_ms
        roof["achieved"] = algo_bytes / (k_ms * 1e-3) / 1e9
        roof["frac"] = roof["achieved"] / hbm_peak
        algo_fma = 4.0 * prof["algo_macs"] / prof["blocks"]
        issued_fma = 4.0 * prof["tile_macs"] / prof["blocks"]
        fp32_peak, fp32_src = 36.3, "fallback: 36.3 TFMA/s measured with tools/bin/microbench on this pool (round 1)"
        try:
            outp = subprocess.run([os.path.join(ROOT, "tools", "bin", "microbench"), "4000"],
                                  capture_output=True, text=True, timeout=60).stdout
            fp32_peak = max(json.loads(ln)["tfma_per_s"] for ln in outp.splitlines() if '"ffma"' in ln)
            fp32_src = "tools/bin/microbench ffma, measured in this run"
        except Exception:  # noqa: BLE001
            pass
        roof["fp32"] = {"bound": "fp32_fma", "achieved": algo_fma / (k_ms * 1e-3) / 1e12,
                        "issued": issued_fma / (k_ms * 1e-3) / 1e12, "peak": fp32_peak, "unit": "TFMA/s",
                        "frac": algo_fma / (k_ms * 1e-3) / 1e12 / fp32_peak, "peak_source": fp32_src,
                        "step_level": {"ms_per_block": ms_per_block,
                                       "achieved": algo_fma / (ms_per_block * 1e-3) / 1e12,
                                       "frac": algo_fma / (ms_per_block * 1e-3) / 1e12 / fp32_peak,
                                       "note": "whole pipelined step (consecutive blocks overlap on alternating compute "
                                               "streams): algorithmic FMAs of a block / device time per block"},
                        "note": "this path is bound by the FP32 FMA pipe, not HBM (DESIGN.md section 4); kernel_ms is "
                                "the kernel alone (non-overlapped pass, CUDA events on its stream)"}
        # what actually binds, in one place: neither HBM nor the tensor pipe but the FP32 FMA pipe -- and of that, the
        # share a shared-memory-fed FFMA loop can reach at all: this kernel's inner loop alone on data already in shared
        # memory, measured in this run (tools/tilebench.cu; all 20 tile shapes: profiles/r2_tilebench.jsonl)
        ceiling, ceiling_src = None, "tools/bin/tilebench not available"
        try:
            outp = subprocess.run([os.path.join(ROOT, "tools", "bin", "tilebench"), "400", "prod"],
                                  capture_output=True, text=True, timeout=60).stdout
            ceiling = max(json.loads(ln)["tfma_per_s"] for ln in outp.splitlines() if '"cur_16x4x8_scalar"' in ln) / fp32_peak
            ceiling_src = "tools/bin/tilebench 400 prod, measured in this run, / the microbench peak"
        except Exception:  # noqa: BLE001
            pass
        roof["binding"] = {"pipe": "fp32_fma", "frac_kernel_alone": roof["fp32"]["frac"],
                           "frac_step": roof["fp32"]["step_level"]["frac"],
                           "loop_ceiling_frac": ceiling, "loop_ceiling_source": ceiling_src,
                           "note": "loop_ceiling = the tiled kernel's inner loop with its operands already in shared "
                                   "memory (no TMA, barriers, epilogue) on all SMs; the step runs on the SMs left of the "
                                   "oscillator partition"}
    roof["step_kernels_ms"] = {k: prof[f"{k}_ms"] / max(prof[f"{k}_launches"], 1)
                               for k in ("convert", "phase", "fir_tile", "fir_long", "fir_generic")}

    launches_per_block = sum(1 for k in ("convert", "phase", "fir_tile", "fir_generic") if prof[f"{k}_launches"] > 0)
    launches_per_block += 2 if prof["fir_long_launches"] > 0 else 0
    ver = main_leg["verified"]
    line = {"metric": "IQ MS/s in", "value": main_leg["value"], "unit": "MS/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_max / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
            "verified": ver["ok"], "verification": ver,
            "e2e": main_leg.get("e2e"), "gpu_launches": launches_per_block * blocks,
            "client_msps": main_leg["value"] * len(wl["plan"]),
            "realtime_clients_per_gpu": int(main_leg["value"] / world * len(wl["plan"]) * 1e6 / wl["fs"]),
            "clocks": clocks, "roofline": roof,
            "engine": {"kernels_used": main_leg["kinds"], "taps_len": sorted({len(t) for t in main_leg["tapsets"].values()}),
                       "sm_partition": ("off (--no-partition)" if args.no_partition else
                                        f"{main_leg['partition_sms']} SMs reserved for the oscillator pre-pass (green contexts), "
                                        "FIR on the others" if main_leg.get("partition_sms") else
                                        "offered (XLG_SM_PARTITION) and declined for this layout: the oscillator chain is short "
                                        "enough to share SMs with the FIR, which keeps all of them"),
                       "block_latency_us": main_leg["block_latency_us"], "host": main_leg["host"], "numa": numa}}
    if legs:
        line["legs"] = legs
    numa_unbind()  # the CPU legs below are entitled to every host core
    if not args.no_cpu and world == 1:
        try:
            line["cpu_baseline"] = cpu_arm(wl, blocks=320, warmup_blocks=16)
        except Exception as ex:  # noqa: BLE001  (the GPU number stands on its own)
            line["cpu_baseline"] = {"error": repr(ex)}
    if not args.no_dropin and world == 1 and wl["fmt"] == "cu8" and args.taps == "default" and wl["name"] in ("cfg2",):
        try:
            line["e2e_dropin"] = dropin_leg(wl)
        except Exception as ex:  # noqa: BLE001
            line["e2e_dropin"] = {"error": repr(ex)}
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
