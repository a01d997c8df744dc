#!/usr/bin/env python
"""bench.py -- headline benchmark of libdeflate_b200 (contract in the task brief, section 4).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference]
                    [--workload roundtrip|decompress] [--chunks C] [--chunk-size B]

Workload (BASELINE.json configs[1]): a batch of 65 536 x 64 KiB synthetic text-like
chunks PER GPU (weak scaling; configs[4] is the same shape at 8 GPUs), gzip level 6
compress followed by gzip decompress of what was just produced.  A "step" is one pass
of that round trip over the batch.  metric = MB/s of UNCOMPRESSED bytes through the
whole round trip (ref: programs/benchmark.c:530-535, programs/test_util.c:197-200).
`--workload decompress` is BASELINE.json configs[2]: raw-DEFLATE decompress-only of the
REFERENCE's own level-6 streams of the same chunks (the north-star roofline kernel).

value  = kernel-path throughput, inputs resident in HBM, CUDA events on the launching
         stream, max over ranks, inputs (4 GiB/GPU) far larger than L2.
e2e    = same metric through libdeflate_b200_*_batch_host with pinned HOST buffers
         (H2D of the inputs and D2H of the results inside the timed region).
roofline / cpu_baseline: see DESIGN.md section "Measurement".
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CHUNK_DEFAULT = 65536
NCHUNKS_DEFAULT = 65536
LEVEL = 6
SYNTH_SO = os.path.join(ROOT, "bench", "libsynth.so")
CPUB_SO = os.path.join(ROOT, "oracle", "_ref", "libcpubench.so")
KIND = {"crc32": 0, "adler32": 1, "inflate": 2, "verify": 3, "deflate": 4, "resolve": 5}


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, gpu_index):
        self.rows = []
        self.proc = None
        self.idx = gpu_index

    def start(self):
        q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + q, "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def dist_env():
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    return rank, world, local


def load_synth():
    if not os.path.exists(SYNTH_SO):
        subprocess.check_call(["gcc", "-O2", "-fPIC", "-shared", "-pthread", "-o", SYNTH_SO, os.path.join(ROOT, "bench", "synth.c"), "-lm"])
    l = ctypes.CDLL(SYNTH_SO)
    l.synth_fill.restype = None
    l.synth_fill.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_size_t, ctypes.c_size_t, ctypes.c_int, ctypes.c_int]
    return l


def load_cpub():
    """oracle/_ref harness around the UNMODIFIED reference (bench-only use of oracle/)."""
    if not os.path.exists(CPUB_SO):
        return None
    l = ctypes.CDLL(CPUB_SO)
    V, S = ctypes.c_void_p, ctypes.c_size_t
    l.cpub_compress.restype = ctypes.c_double
    l.cpub_compress.argtypes = [ctypes.c_int, ctypes.c_int, V, S, S, V, S, V, ctypes.c_int, ctypes.POINTER(ctypes.c_int)]
    l.cpub_decompress.restype = ctypes.c_double
    l.cpub_decompress.argtypes = [ctypes.c_int, V, V, V, S, V, S, ctypes.c_int, ctypes.POINTER(ctypes.c_int)]
    l.cpub_checksum.restype = ctypes.c_double
    l.cpub_checksum.argtypes = [ctypes.c_int, V, S, S, V, ctypes.c_int]
    return l


def cpu_quota():
    """CPUs this container may actually use: min(affinity mask, cgroup cpu.max quota)."""
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            f = open(path).read().split()
            if path.endswith("cpu.max"):
                if f[0] != "max":
                    n = min(n, max(1, int(int(f[0]) / int(f[1]) + 0.5)))
            else:
                q = int(f[0])
                per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if q > 0:
                    n = min(n, max(1, int(q / per + 0.5)))
            break
        except Exception:
            continue
    return n


def host_threads():
    """Threads for the CPU reference arm: one per usable CPU (more only gets throttled by the quota)."""
    return cpu_quota()


def cpu_roundtrip(cpub, fmt, level, host_in, chunk, n, threads, want_streams=False):
    """Reference compress + decompress of n chunks on `threads` host threads.
    Returns (t_compress, t_decompress, compressed_bytes, streams?)"""
    stride = chunk + 5 * ((chunk + 4999) // 5000) + 18
    comp = (ctypes.c_uint8 * (stride * n))()
    sizes = (ctypes.c_size_t * n)()
    fails = ctypes.c_int(0)
    tc = cpub.cpub_compress(fmt, level, host_in, chunk, n, comp, stride, sizes, threads, ctypes.byref(fails))
    assert fails.value == 0, "reference compress failed"
    offs = (ctypes.c_size_t * n)(*[i * stride for i in range(n)])
    out = (ctypes.c_uint8 * (chunk * n))()
    td = cpub.cpub_decompress(fmt, comp, offs, sizes, n, out, chunk, threads, ctypes.byref(fails))
    assert fails.value == 0, "reference decompress failed"
    total = sum(sizes)
    if want_streams:
        return tc, td, total, (comp, stride, sizes)
    return tc, td, total, None


def run_reference(args):
    """--impl reference: the reference's own CPU implementation on the host cores, on the SAME
    batch shape as the GPU arm (identical `config`), bounded only if the host is too slow for it."""
    rank, world, local = dist_env()
    if rank != 0:
        return
    cpub = load_cpub()
    if cpub is None:
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/libcpubench.so not built (needs /root/reference at build time)"}))
        return
    synth = load_synth()
    threads = host_threads()
    chunk = args.chunk_size
    n = args.chunks
    buf = (ctypes.c_uint8 * (n * chunk))()
    synth.synth_fill(buf, chunk, 0, n, getattr(args, "data_class", 0), threads)
    fmt = 2 if args.workload == "roundtrip" else 0
    times = []
    ratio = None
    bounded = None
    for it in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        tc, td, total, streams = cpu_roundtrip(cpub, fmt, LEVEL, buf, chunk, n, threads, want_streams=(args.workload == "decompress"))
        ratio = total / float(n * chunk)
        t = (tc + td) if args.workload == "roundtrip" else td
        if it >= args.warmup:
            times.append((t, tc, td, n))
        if it == 0:
            # a host with very few usable CPUs: keep the whole run within a few minutes by sampling the batch
            per_pass = time.perf_counter() - t0
            budget = 180.0 / (args.warmup + args.steps)
            while per_pass > budget and n > 1024:
                n //= 2
                per_pass /= 2
                bounded = n
    tsum = sum(t[0] for t in times)
    nbytes = sum(t[3] for t in times) * chunk
    value = nbytes / 1e6 / tsum
    cfg = workload_config(args)
    if bounded:
        cfg["reference_sample"] = "first %d chunks per step (host too slow for the full batch within the time budget)" % bounded
    line = {
        "impl": "reference",
        "metric": metric_name(args), "value": round(value, 2), "unit": "MB/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": round(1e3 * tsum / len(times), 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": round(value, 2), "unit": "MB/s", "cores": threads, "host_cpus_online": os.cpu_count(), "cpu_quota": cpu_quota(), "kind": "reference",
                         "per_thread_MBps": round(value / threads, 2),
                         "sample": "%d x %d B chunks per step, gzip L%d compress+decompress with oracle/_ref (unmodified libdeflate), %d threads"
                                   % (n, chunk, LEVEL, threads) if args.workload == "roundtrip" else
                                   "%d x %d B chunks per step, raw DEFLATE decompress of reference L%d streams, %d threads" % (n, chunk, LEVEL, threads),
                         "compress_MBps": round(nbytes / 1e6 / sum(t[1] for t in times), 2),
                         "decompress_MBps": round(nbytes / 1e6 / sum(t[2] for t in times), 2),
                         "ratio": round(ratio, 4)},
        "e2e": {"value": round(value, 2), "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def metric_name(args):
    if args.workload == "decompress":
        return "MB/s raw DEFLATE decompress (batched 64 KiB chunks, reference L6 streams)"
    return "MB/s compress+decompress (batched 64 KiB chunks)"


def workload_config(args, n_override=None):
    n = n_override if n_override is not None else args.chunks
    if args.workload == "decompress":
        w = "batch of %d x %d B synthetic text chunks per GPU, raw DEFLATE decompress-only of the reference's level-%d streams" % (n, args.chunk_size, LEVEL)
    else:
        w = "batch of %d x %d B synthetic text chunks per GPU, gzip level %d compress+decompress" % (n, args.chunk_size, LEVEL)
    return {"workload": w, "chunks_per_gpu": n, "chunk_bytes": args.chunk_size, "level": LEVEL,
            "format": "raw" if args.workload == "decompress" else "gzip",
            "l2_policy": "inputs (%.1f GiB per GPU) are far larger than the 126 MB L2; no explicit flush" % (n * args.chunk_size / 2.0**30),
            "parallelism": "independent chunk shards per GPU, no data-path collective (the single-origin NCCL scatter/gather run of the same batch is reported under single_origin when N > 1)"}


class DeviceBatch:
    """Device-resident batch: a slab (owned, or a view of another batch's slab) plus device arrays
    of pointers/sizes."""

    def __init__(self, ctx, n, stride, slab=None):
        import numpy as np
        self.ctx, self.n, self.stride = ctx, n, stride
        l = ctx.l
        self.own = slab is None
        self.slab = l.libdeflate_b200_device_malloc(ctx.h, n * stride + 256) if slab is None else slab
        self.d_ptrs = l.libdeflate_b200_device_malloc(ctx.h, 8 * n)
        self.d_sizes = l.libdeflate_b200_device_malloc(ctx.h, 8 * n)
        assert self.slab and self.d_ptrs and self.d_sizes, "device_malloc failed"
        ptrs = (self.slab + np.arange(n, dtype=np.uint64) * np.uint64(stride)).astype(np.uint64)
        self._keep = ptrs
        ctx._check(l.libdeflate_b200_memcpy_h2d(ctx.h, self.d_ptrs, ptrs.ctypes.data, 8 * n), "h2d")
        ctx.sync()

    def set_sizes(self, sizes_np):
        self._keep_s = sizes_np
        self.ctx._check(self.ctx.l.libdeflate_b200_memcpy_h2d(self.ctx.h, self.d_sizes, sizes_np.ctypes.data, 8 * self.n), "h2d")
        self.ctx.sync()

    def free(self):
        for p in ((self.slab,) if self.own else ()) + (self.d_ptrs, self.d_sizes):
            self.ctx.l.libdeflate_b200_device_free(self.ctx.h, p)


def timed_steps(ctx, l, step, steps, warmup, barrier=None, clocks=None):
    """W untimed steps, then K steps between two CUDA events on the launching stream; per-kernel
    device time from the library's own event pairs around every launch in the same region."""
    for _ in range(warmup):
        step()
    ctx.sync()
    l.libdeflate_b200_ctx_set_profiling(ctx.h, 1)
    l.libdeflate_b200_kernel_time_reset(ctx.h)
    launches0 = ctx.launches
    if barrier:
        barrier()
    ctx.sync()
    if clocks:
        clocks.start()
    l.libdeflate_b200_timer_start(ctx.h)
    for _ in range(steps):
        step()
    ms = max(l.libdeflate_b200_timer_stop_ms(ctx.h), 1e-9)
    ctx.sync()
    if barrier:
        barrier()
    clk = clocks.stop() if clocks else None
    launches = ctx.launches - launches0
    ktime = {}
    for name, k in KIND.items():
        cnt = ctypes.c_uint64(0)
        t = l.libdeflate_b200_kernel_time_ms(ctx.h, k, ctypes.byref(cnt))
        ktime[name] = (t, cnt.value)
    l.libdeflate_b200_ctx_set_profiling(ctx.h, 0)
    return ms, ktime, launches, clk


def load_traffic(key):
    try:
        return json.load(open(os.path.join(ROOT, "profiles", "dram_traffic.json"))).get(key, {})
    except Exception:
        return {}


def roofline_entry(kernels, ms_total, launches, alg_bytes, traffic_db, traffic_key, peak, peak_src):
    """achieved = algorithmic bytes per launch / average duration of the named kernel(s)."""
    if not launches or ms_total <= 0:
        return None
    per = ms_total / launches / 1e3
    ach = alg_bytes / per / 1e9
    tr = 0.0
    for k in kernels:
        v = traffic_db.get(k, {}).get("dram_bytes_per_launch")
        if not v:
            tr = None
            break
        tr += v
    return {"kernel": " + ".join(kernels), "bound": "hbm", "achieved": round(ach, 2), "peak": peak, "unit": "GB/s",
            "frac": round(ach / peak, 4), "traffic": int(tr) if tr else None,
            "traffic_over_algorithmic": round(tr / alg_bytes, 3) if tr else None,
            "traffic_source": ("profiles/dram_traffic.json[%s] (ncu dram__bytes_read+write of this build, same configuration)" % traffic_key) if tr else None,
            "peak_source": peak_src,
            "avg_launch_ms": round(per * 1e3, 4), "algorithmic_bytes_per_launch": int(alg_bytes)}


def run_b200(args):
    import numpy as np
    import libdeflate_b200 as ldb
    from libdeflate_b200 import shard
    rank, world, local = shard.dist_env()
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist_mod
        torch.cuda.set_device(local)
        # NCCL announces its version on stdout when the first communicator comes up; the contract is ONE
        # JSON line on stdout, so stdout points at stderr until that has happened
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist_mod.init_process_group("nccl", device_id=torch.device("cuda", local))
            dist_mod.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
        dist = dist_mod
    red = shard.Reducer(dist, "cuda" if dist else "cpu")
    barrier, allmax, allsum = red.barrier, red.max, red.sum

    l = ldb.lib()
    if l.libdeflate_b200_device_count() <= local:
        raise SystemExit("bench.py: no CUDA device for local rank %d -- libdeflate_b200 has no CPU fallback" % local)
    ctx = ldb.Context(local)
    synth = load_synth()
    cpub = load_cpub()
    threads = max(1, host_threads() // max(1, world))
    n, chunk = args.chunks, args.chunk_size
    fmt = ldb.GZIP if args.workload == "roundtrip" else ldb.RAW
    bound = l.libdeflate_gzip_compress_bound(None, chunk)
    cstride = (bound + 15) & ~15
    peak, peak_src = load_peaks()

    # ---- inputs: synthetic chunks generated on the host (pinned), then resident in HBM ----
    pin_in = l.libdeflate_b200_pinned_malloc(n * chunk)
    assert pin_in, "pinned_malloc failed"
    first_chunk, _ = shard.shard_range(rank, world, n)
    synth.synth_fill(pin_in, chunk, first_chunk, n, getattr(args, "data_class", 0), threads)
    d_in = DeviceBatch(ctx, n, chunk)
    ctx._check(l.libdeflate_b200_memcpy_h2d(ctx.h, d_in.slab, pin_in, n * chunk), "h2d")
    d_in.set_sizes(np.full(n, chunk, dtype=np.uint64))
    d_comp = DeviceBatch(ctx, n, cstride)
    d_comp.set_sizes(np.full(n, cstride, dtype=np.uint64))      # avail for compress
    d_out = DeviceBatch(ctx, n, chunk)
    d_out.set_sizes(np.full(n, chunk, dtype=np.uint64))
    d_csz = l.libdeflate_b200_device_malloc(ctx.h, 8 * n)          # compressed sizes (device)
    d_aout = l.libdeflate_b200_device_malloc(ctx.h, 8 * n)
    d_res = l.libdeflate_b200_device_malloc(ctx.h, 4 * n)

    def load_reference_streams():
        """the reference's own L6 raw streams for the same chunks (SURVEY.md section 8d) -> d_comp / d_csz"""
        assert cpub is not None, "the decompress workload needs oracle/_ref (prebuilt from /root/reference)"
        comp = (ctypes.c_uint8 * (cstride * n))()
        sizes = (ctypes.c_size_t * n)()
        fails = ctypes.c_int(0)
        cpub.cpub_compress(0, 6, pin_in, chunk, n, comp, cstride, sizes, threads, ctypes.byref(fails))
        assert fails.value == 0
        ctx._check(l.libdeflate_b200_memcpy_h2d(ctx.h, d_comp.slab, comp, cstride * n), "h2d")
        cs = np.frombuffer(sizes, dtype=np.uint64).copy()
        ctx._check(l.libdeflate_b200_memcpy_h2d(ctx.h, d_csz, cs.ctypes.data, 8 * n), "h2d")
        ctx.sync()
        return cs

    def decompress_step(f):
        ctx._check(l.libdeflate_b200_decompress_batch(ctx.h, f, 0, d_comp.d_ptrs, d_csz, d_out.d_ptrs, d_out.d_sizes, None, d_aout, d_res, n), "decompress_batch")

    def check_outputs(what, verdicts=True):
        if verdicts:
            res = np.empty(n, dtype=np.int32)
            aout = np.empty(n, dtype=np.uint64)
            ctx._check(l.libdeflate_b200_memcpy_d2h(ctx.h, res.ctypes.data, d_res, 4 * n), "d2h")
            ctx._check(l.libdeflate_b200_memcpy_d2h(ctx.h, aout.ctypes.data, d_aout, 8 * n), "d2h")
            ctx.sync()
            assert (res == 0).all(), "%s: decompress verdicts not all SUCCESS: %s" % (what, np.unique(res, return_counts=True))
            assert (aout == chunk).all(), "%s: decompressed sizes wrong" % what
        # checksum of checksums over every chunk (device CRC-32 of outputs vs inputs)
        d_c1 = l.libdeflate_b200_device_malloc(ctx.h, 4 * n)
        d_c2 = l.libdeflate_b200_device_malloc(ctx.h, 4 * n)
        ctx._check(l.libdeflate_b200_crc32_batch(ctx.h, d_in.d_ptrs, d_in.d_sizes, None, d_c1, n), "crc")
        ctx._check(l.libdeflate_b200_crc32_batch(ctx.h, d_out.d_ptrs, d_out.d_sizes, None, d_c2, n), "crc")
        c1 = np.empty(n, dtype=np.uint32)
        c2 = np.empty(n, dtype=np.uint32)
        ctx._check(l.libdeflate_b200_memcpy_d2h(ctx.h, c1.ctypes.data, d_c1, 4 * n), "d2h")
        ctx._check(l.libdeflate_b200_memcpy_d2h(ctx.h, c2.ctypes.data, d_c2, 4 * n), "d2h")
        ctx.sync()
        l.libdeflate_b200_device_free(ctx.h, d_c1)
        l.libdeflate_b200_device_free(ctx.h, d_c2)
        assert (c1 == c2).all(), "%s: round trip mismatch (device CRC of output != input)" % what
        return c2

    ref_ratio = None
    csz_ref = None
    if args.workload == "decompress":
        csz_ref = load_reference_streams()
        ref_ratio = float(csz_ref.sum()) / (n * chunk)

    def step():
        if args.workload == "roundtrip":
            ctx._check(l.libdeflate_b200_compress_batch(ctx.h, fmt, LEVEL, d_in.d_ptrs, d_in.d_sizes, d_comp.d_ptrs, d_comp.d_sizes, d_csz, n), "compress_batch")
        decompress_step(fmt)

    # ---- kernel-path timing of the main workload --------------------------------------------
    clocks = ClockSampler(local) if rank == 0 else None
    ms, ktime, launches, clk = timed_steps(ctx, l, step, args.steps, args.warmup, barrier, clocks)
    ms_max = max(allmax(ms), 1e-9)

    # ---- verification (outside the timed region) ----------------------------------------
    c2 = check_outputs("main workload")
    csz = np.empty(n, dtype=np.uint64)
    ctx._check(l.libdeflate_b200_memcpy_d2h(ctx.h, csz.ctypes.data, d_csz, 8 * n), "d2h")
    ctx.sync()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ctx, l, n, chunk, cstride, csz, d_comp, d_out, d_aout, d_res,
                     args.workload == "roundtrip")
    assert (csz > 0).all(), "a chunk did not fit its compress bound"
    # bit-exact byte comparison with the host originals on every 64th chunk
    samp = np.arange(0, n, 64)
    host_in = np.ctypeslib.as_array(ctypes.cast(pin_in, ctypes.POINTER(ctypes.c_uint8)), shape=(n * chunk,))
    tmp = np.empty(chunk, dtype=np.uint8)
    import zlib
    for i in samp[:256]:
        ctx._check(l.libdeflate_b200_memcpy_d2h(ctx.h, tmp.ctypes.data, d_out.slab + int(i) * chunk, chunk), "d2h")
        ctx.sync()
        assert np.array_equal(tmp, host_in[int(i) * chunk:(int(i) + 1) * chunk]), "byte mismatch in chunk %d" % i
        assert zlib.crc32(tmp.tobytes()) == int(c2[i]), "device CRC-32 disagrees with zlib on chunk %d" % i
    ratio = float(csz.sum()) / (n * chunk)
    comp_bytes = float(csz.sum())

    # ---- e2e: host buffers through the public *_batch_host calls -------------------------
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(args, ctx, l, ldb, pin_in, n, chunk, fmt, cstride, barrier, allmax, d_comp if args.workload == "decompress" else None, csz)

    # ---- cpu baseline (rank 0, N=1 only): bounded sample of the same workload ------------
    cpu_baseline = None
    if rank == 0 and world == 1 and cpub is not None and not args.no_cpu:
        ht = host_threads()
        ns = min(n, max(1024, 2048 * ht))
        tc, td, total, _ = cpu_roundtrip(cpub, 2 if args.workload == "roundtrip" else 0, LEVEL, pin_in, chunk, ns, ht)
        t = (tc + td) if args.workload == "roundtrip" else td
        cpu_baseline = {"value": round(ns * chunk / 1e6 / t, 2), "unit": "MB/s", "cores": ht, "host_cpus_online": os.cpu_count(), "cpu_quota": cpu_quota(), "kind": "reference",
                        "per_thread_MBps": round(ns * chunk / 1e6 / t / ht, 2),
                        "sample": "first %d chunks of the same batch, one pass, oracle/_ref (unmodified libdeflate 1.25, -O2) on %d host threads" % (ns, ht),
                        "compress_MBps": round(ns * chunk / 1e6 / tc, 2), "decompress_MBps": round(ns * chunk / 1e6 / td, 2),
                        "ratio": round(total / float(ns * chunk), 4)}
        n1 = min(n, 256)
        tc1, td1, _, _ = cpu_roundtrip(cpub, 2 if args.workload == "roundtrip" else 0, LEVEL, pin_in, chunk, n1, 1)
        cpu_baseline["one_thread_compress_MBps"] = round(n1 * chunk / 1e6 / tc1, 2)
        cpu_baseline["one_thread_decompress_MBps"] = round(n1 * chunk / 1e6 / td1, 2)

    # ---- rooflines of the main workload ----------------------------------------------------
    steps = args.steps
    total_unc = allsum(float(n * chunk))
    value = total_unc * steps / 1e6 / (ms_max / 1e3)
    # algorithmic bytes per launch (DESIGN.md): inflate = compressed in + uncompressed out over the
    # decode + resolve pair; deflate = uncompressed in + compressed out
    alg = n * chunk + comp_bytes
    tkey = "%s_L%d_%dx%d" % (args.workload, LEVEL, n, chunk)
    tdb = load_traffic(tkey)
    INF = ["ldb_inflate_decode_kernel", "ldb_inflate_resolve_kernel"]
    t_inf = ktime["inflate"][0] + ktime["resolve"][0]
    r_inf = roofline_entry(INF, t_inf, ktime["inflate"][1], alg, tdb, tkey, peak, peak_src)
    if r_inf:
        r_inf["decode_ms"] = round(ktime["inflate"][0] / max(1, ktime["inflate"][1]), 4)
        r_inf["resolve_ms"] = round(ktime["resolve"][0] / max(1, ktime["resolve"][1]), 4)
    r_def = roofline_entry(["ldb_deflate_lz_kernel"], ktime["deflate"][0], ktime["deflate"][1], alg, tdb, tkey, peak, peak_src)
    dominant = r_def if (r_def and ktime["deflate"][0] >= t_inf) else r_inf

    # ---- the other BASELINE configurations, short legs (N=1 only) ----------------------------
    extra = None
    if world == 1 and not args.no_extra and args.workload == "roundtrip" and chunk == CHUNK_DEFAULT:
        extra = {}
        # (configs[2]) raw DEFLATE decompress-only of the REFERENCE's L6 streams: the north-star roofline run
        if cpub is not None:
            cs = load_reference_streams()
            k = max(3, min(args.steps, 10))
            ms_d, kt_d, _, _ = timed_steps(ctx, l, lambda: decompress_step(ldb.RAW), k, 3)
            check_outputs("decompress leg")
            alg_d = n * chunk + float(cs.sum())
            dkey = "decompress_L6_%dx%d" % (n, chunk)
            rd = roofline_entry(INF, kt_d["inflate"][0] + kt_d["resolve"][0], kt_d["inflate"][1], alg_d, load_traffic(dkey), dkey, peak, peak_src)
            if rd:
                rd["decode_ms"] = round(kt_d["inflate"][0] / k, 4)
                rd["resolve_ms"] = round(kt_d["resolve"][0] / k, 4)
            leg = {"config": "configs[2]: %d x %d B raw DEFLATE decompress-only, the reference's own level-6 streams" % (n, chunk),
                   "value": round(n * chunk * k / 1e6 / (ms_d / 1e3), 2), "unit": "MB/s", "steps": k, "warmup": 3, "ms_per_step": round(ms_d / k, 4),
                   "ratio_reference_L6": round(float(cs.sum()) / (n * chunk), 4), "roofline": rd}
            if rank == 0 and not args.no_cpu:
                ht = host_threads()
                ns = min(n, max(1024, 2048 * ht))
                _, td, _, _ = cpu_roundtrip(cpub, 0, 6, pin_in, chunk, ns, ht)
                leg["cpu_baseline"] = {"value": round(ns * chunk / 1e6 / td, 2), "unit": "MB/s", "cores": ht, "kind": "reference",
                                       "per_thread_MBps": round(ns * chunk / 1e6 / td / ht, 2),
                                       "sample": "first %d chunks, one raw-DEFLATE decompress pass of the reference on %d host threads" % (ns, ht)}
            extra["decompress_reference_streams"] = leg
            r_inf_north = rd
        else:
            r_inf_north = None
        # standalone checksum kernels over the input batch
        d_sum = l.libdeflate_b200_device_malloc(ctx.h, 4 * n)
        for kind, fn in (("crc32", l.libdeflate_b200_crc32_batch), ("adler32", l.libdeflate_b200_adler32_batch)):
            ms_c, kt_c, _, _ = timed_steps(ctx, l, lambda: ctx._check(fn(ctx.h, d_in.d_ptrs, d_in.d_sizes, None, d_sum, n), kind), 10, 3)
            rc = roofline_entry(["ldb_%s_kernel" % kind], kt_c[kind][0], kt_c[kind][1], float(n * chunk), {}, "", peak, peak_src)
            extra[kind] = {"config": "%d x %d B, one %s per chunk" % (n, chunk, kind), "value": round(n * chunk * 10 / 1e6 / (ms_c / 1e3), 2), "unit": "MB/s",
                           "ms_per_step": round(ms_c / 10, 4), "roofline": rc}
        l.libdeflate_b200_device_free(ctx.h, d_sum)
        if cpub is not None and rank == 0 and not args.no_cpu:
            ht = host_threads()
            ns = min(n, 4096 * ht)
            sums = (ctypes.c_uint32 * ns)()
            for kind, isad in (("crc32", 0), ("adler32", 1)):
                t = cpub.cpub_checksum(isad, pin_in, chunk, ns, sums, ht)
                extra[kind]["cpu_baseline"] = {"value": round(ns * chunk / 1e6 / t, 2), "unit": "MB/s", "cores": ht, "kind": "reference"}
        # (configs[3]) level 12, 4096 x 1 MiB: same bytes, 16 chunks fused into one
        if not args.no_l12 and n * chunk >= getattr(args, "l12_min_bytes", 1 << 30):
            n12, c12 = n * chunk >> 20, 1 << 20
            b12 = (l.libdeflate_gzip_compress_bound(None, c12) + 15) & ~15
            if n12 * b12 <= n * cstride:
                v_in = DeviceBatch(ctx, n12, c12, d_in.slab)
                v_in.set_sizes(np.full(n12, c12, dtype=np.uint64))
                v_comp = DeviceBatch(ctx, n12, b12, d_comp.slab)
                v_comp.set_sizes(np.full(n12, b12, dtype=np.uint64))
                v_out = DeviceBatch(ctx, n12, c12, d_out.slab)
                v_out.set_sizes(np.full(n12, c12, dtype=np.uint64))

                def step12():
                    ctx._check(l.libdeflate_b200_compress_batch(ctx.h, ldb.GZIP, 12, v_in.d_ptrs, v_in.d_sizes, v_comp.d_ptrs, v_comp.d_sizes, d_csz, n12), "compress_batch L12")
                    ctx._check(l.libdeflate_b200_decompress_batch(ctx.h, ldb.GZIP, 0, v_comp.d_ptrs, d_csz, v_out.d_ptrs, v_out.d_sizes, None, d_aout, d_res, n12), "decompress_batch L12")
                ms12, kt12, _, _ = timed_steps(ctx, l, step12, 1, 1)
                res12 = np.empty(n12, dtype=np.int32)
                cs12 = np.empty(n12, dtype=np.uint64)
                ctx._check(l.libdeflate_b200_memcpy_d2h(ctx.h, res12.ctypes.data, d_res, 4 * n12), "d2h")
                ctx._check(l.libdeflate_b200_memcpy_d2h(ctx.h, cs12.ctypes.data, d_csz, 8 * n12), "d2h")
                ctx.sync()
                assert (res12 == 0).all() and (cs12 > 0).all(), "level-12 leg failed"
                # bytes: the 1 MiB views alias the 64 KiB batch, so output == input chunk for chunk
                check_outputs("level-12 leg", verdicts=False)
                alg12 = n12 * c12 + float(cs12.sum())
                leg = {"config": "configs[3]: %d x %d B gzip level 12 compress + decompress" % (n12, c12),
                       "value": round(n12 * c12 / 1e6 / (ms12 / 1e3), 2), "unit": "MB/s", "steps": 1, "warmup": 1, "ms_per_step": round(ms12, 2),
                       "kernel_ms_per_step": {k: round(v[0], 3) for k, v in kt12.items() if v[1]},
                       "ratio": round(float(cs12.sum()) / (n12 * c12), 4),
                       "roofline": roofline_entry(["ldb_deflate_lz_kernel"], kt12["deflate"][0], kt12["deflate"][1], alg12, {}, "", peak, peak_src)}
                if cpub is not None and rank == 0 and not args.no_cpu:
                    ht = host_threads()
                    ns = min(n12, max(ht, 16))
                    hostbuf = ctypes.cast(pin_in, ctypes.POINTER(ctypes.c_uint8))
                    comp = (ctypes.c_uint8 * (b12 * ns))()
                    sizes = (ctypes.c_size_t * ns)()
                    fails = ctypes.c_int(0)
                    t = cpub.cpub_compress(2, 12, hostbuf, c12, ns, comp, b12, sizes, ht, ctypes.byref(fails))
                    leg["cpu_baseline"] = {"compress_MBps": round(ns * c12 / 1e6 / t, 2), "cores": ht, "kind": "reference", "ratio": round(sum(sizes) / float(ns * c12), 4),
                                           "sample": "first %d x 1 MiB chunks, one level-12 gzip compress pass of the reference on %d host threads" % (ns, ht)}
                extra["level12_1MiB"] = leg
                for v in (v_in, v_comp, v_out):
                    v.free()
    else:
        r_inf_north = None

    # ---- BASELINE configs[4]: the same round trip when ONE rank owns the whole batch (NCCL data plane) ----
    single_origin = None
    if world > 1 and not args.no_origin and args.workload == "roundtrip":
        import torch
        for b in (d_in, d_comp, d_out):
            b.free()
        for p_ in (d_csz, d_aout, d_res):
            l.libdeflate_b200_device_free(ctx.h, p_)
        dev = torch.device("cuda", local)
        n_total = n * world
        rt = shard.OriginRoundTrip(ctx, dist, dev, n_total, chunk, fmt, LEVEL, stages=8)
        root_in = None
        if rank == 0:
            root_in = torch.empty(n_total * chunk, dtype=torch.uint8, device=dev)
            for r in range(world):        # the batch of the pre-sharded run, rank by rank, through the one pinned buffer
                synth.synth_fill(pin_in, chunk, r * n, n, getattr(args, "data_class", 0), threads)
                ctx._check(l.libdeflate_b200_memcpy_h2d(ctx.h, root_in.data_ptr() + r * n * chunk, pin_in, n * chunk), "h2d")
                ctx.sync()
        so_steps = max(1, min(args.steps, 2))
        info = rt.step(root_in)           # warm-up (NCCL channels, scratch)
        barrier()
        ctx.sync()
        l.libdeflate_b200_timer_start(ctx.h)
        for _ in range(so_steps):
            info = rt.step(root_in)
        ms_so = l.libdeflate_b200_timer_stop_ms(ctx.h)
        barrier()
        ms_so = allmax(ms_so)
        ok = bool((rt.res[:rt.n] == 0).all().item())
        if rank == 0:
            ok = ok and bool(torch.equal(rt.out_all, root_in))
        ok_all = allsum(1.0 if ok else 0.0)
        single_origin = {"config": "configs[4]: %d x %d B gzip level %d round trip, the whole batch on rank 0, %d GPUs" % (n_total, chunk, LEVEL, world),
                         "value": round(n_total * chunk * so_steps / 1e6 / (ms_so / 1e3), 2), "unit": "MB/s", "steps": so_steps, "warmup": 1,
                         "ms_per_step": round(ms_so / so_steps, 3),
                         "parallelism": "NCCL scatter/gather: grouped ncclSend/ncclRecv of sub-batches root<->ranks overlapped with the kernels, device-side packing, all_gather of byte totals",
                         "comm_nranks_ok": int(ok_all) == world, "verified": "all ranks SUCCESS; gathered output == input on the root (torch.equal)",
                         "root_nvlink_bytes_per_step": info["nvlink_bytes"], "compressed_bytes_per_step": info["compressed_bytes_total"],
                         "timing": "CUDA events on each rank's stream around the steps, max over ranks"}
        assert int(ok_all) == world, "single-origin round trip failed verification"

    line = {
        "metric": metric_name(args), "value": round(value, 2), "unit": "MB/s", "n_gpus": world,
        "steps": steps, "warmup": args.warmup, "ms_per_step": round(ms_max / steps, 4),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic" if getattr(args, "data_class", 0) == 0 else "synthetic (class %d of bench/synth.c, not the headline corpus)" % args.data_class,
        "config": workload_config(args),
        "roofline": dominant, "roofline_inflate": r_inf_north or r_inf, "roofline_deflate": r_def,
        "kernel_ms_per_step": {k: round(v[0] / steps, 4) for k, v in ktime.items() if v[1]},
        "ratio": round(ratio, 4), "ratio_reference_L6": ref_ratio,
        "cpu_baseline": cpu_baseline, "e2e": e2e, "gpu_launches": int(launches), "clocks": clk,
        "extra": extra, "single_origin": single_origin,
        "verified": "all %d chunks: verdict SUCCESS, size, device CRC-32(out)==CRC-32(in); %d chunks byte-compared + zlib CRC" % (n, min(256, len(samp))),
    }
    if rank == 0:
        print(json.dumps(line))
    if dist:
        dist.destroy_process_group()


DUMP_PER_CHUNK_BYTES = 12_000_000     # four float64 values per chunk listed
DUMP_SAMPLE_BYTES = 48_000_000        # float32 bytes of the sampled chunks
DUMP_SAMPLE_CHUNKS = 96


def dump_outputs(out_dir, ctx, l, n, chunk, cstride, csz, d_comp, d_out, d_aout, d_res, compressed):
    """What the last timed step handed back, as .npy files of float64 (per-chunk values) and float32 (bytes),
    about 60 MB at most whatever the batch shape:
      decompress_results, decompressed_sizes and, when the step compressed, compressed_sizes: one value per
          chunk named in chunk_index -- every chunk, or a fixed, seeded sample once the batch is too large for
          DUMP_PER_CHUNK_BYTES;
      sample_decompressed and, when the step compressed, sample_compressed (the stream zero-padded to its slot):
          the bytes of a fixed, seeded sample of chunks (sample_chunk_index), as many as DUMP_SAMPLE_BYTES holds
          up to 96, and only the leading bytes of each when one chunk alone does not fit.
    With --workload decompress the compressed streams are the reference's, an input of the step, so they are
    not written.  The inputs are the same from run to run, so two builds compare file for file."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(0)

    def sample(count):
        return np.arange(n) if count >= n else np.sort(rng.choice(n, count, replace=False))
    res = np.empty(n, dtype=np.int32)
    aout = np.empty(n, dtype=np.uint64)
    ctx._check(l.libdeflate_b200_memcpy_d2h(ctx.h, res.ctypes.data, d_res, 4 * n), "d2h")
    ctx._check(l.libdeflate_b200_memcpy_d2h(ctx.h, aout.ctypes.data, d_aout, 8 * n), "d2h")
    per = sample(DUMP_PER_CHUNK_BYTES // (8 * 4))
    arrays = {"chunk_index": per, "decompress_results": res[per], "decompressed_sizes": aout[per]}
    row_bytes = 4 * (chunk + (cstride if compressed else 0))
    idx = sample(max(1, min(DUMP_SAMPLE_CHUNKS, DUMP_SAMPLE_BYTES // row_bytes)))
    cap = DUMP_SAMPLE_BYTES // (4 * len(idx) * (2 if compressed else 1))
    out_len, comp_len = min(chunk, cap), min(cstride, cap)
    out = np.empty((len(idx), out_len), dtype=np.uint8)
    comp = np.zeros((len(idx), comp_len), dtype=np.uint8)
    for k, i in enumerate(idx):
        ctx._check(l.libdeflate_b200_memcpy_d2h(ctx.h, out[k].ctypes.data, d_out.slab + int(i) * chunk, out_len), "d2h")
        if compressed:
            ctx._check(l.libdeflate_b200_memcpy_d2h(ctx.h, comp[k].ctypes.data, d_comp.slab + int(i) * cstride,
                                                    min(int(csz[i]), comp_len)), "d2h")
    ctx.sync()
    arrays.update(sample_chunk_index=idx, sample_decompressed=out)
    if compressed:
        arrays.update(compressed_sizes=csz[per], sample_compressed=comp)
    for name, a in arrays.items():
        a = a.astype(np.float32 if name.startswith("sample_") and name != "sample_chunk_index" else np.float64)
        np.save(os.path.join(out_dir, name + ".npy"), a)


def run_e2e(args, ctx, l, ldb, pin_in, n, chunk, fmt, cstride, barrier, allmax, d_comp_ref, csz_ref):
    """Same metric through the host-buffer C-ABI calls a chunk-loop caller would make; pinned host memory on
    both sides.  The compressed side uses the PACKED forms (one buffer + offset table): the device packs the
    bound-sized slots, so only produced bytes cross PCIe."""
    import numpy as np
    try:
        import psutil
        avail = psutil.virtual_memory().available
    except Exception:
        avail = 64 << 30
    ne = n
    while ne > 1024 and ne * (chunk + cstride + chunk) * 2 > avail // 8:
        ne //= 2
    packed_cap = ne * (cstride + 16)
    pin_comp = l.libdeflate_b200_pinned_malloc(packed_cap)
    pin_out = l.libdeflate_b200_pinned_malloc(ne * chunk)
    assert pin_comp and pin_out

    def arr(base, stride, cnt):
        return (base + np.arange(cnt, dtype=np.uint64) * np.uint64(stride)).astype(np.uint64)
    in_ptrs = arr(pin_in, chunk, ne)
    in_sizes = np.full(ne, chunk, dtype=np.uint64)
    out_ptrs = arr(pin_out, chunk, ne)
    out_avail = np.full(ne, chunk, dtype=np.uint64)
    comp_sizes = np.zeros(ne, dtype=np.uint64)
    comp_offs = np.zeros(ne + 1, dtype=np.uint64)
    aout = np.zeros(ne, dtype=np.uint64)
    res = np.zeros(ne, dtype=np.int32)
    if args.workload == "decompress":
        # host copy of the reference streams, packed (16-byte aligned starts) -- outside the timed region
        tmp = l.libdeflate_b200_pinned_malloc(ne * cstride)
        ctx._check(l.libdeflate_b200_memcpy_d2h(ctx.h, tmp, d_comp_ref.slab, ne * cstride), "d2h")
        ctx.sync()
        comp_sizes[:] = csz_ref[:ne]
        comp_offs[1:] = np.cumsum((comp_sizes + np.uint64(15)) & ~np.uint64(15))
        src = np.ctypeslib.as_array(ctypes.cast(tmp, ctypes.POINTER(ctypes.c_uint8)), shape=(ne * cstride,))
        dst = np.ctypeslib.as_array(ctypes.cast(pin_comp, ctypes.POINTER(ctypes.c_uint8)), shape=(packed_cap,))
        for i in range(ne):
            o, z = int(comp_offs[i]), int(comp_sizes[i])
            dst[o:o + z] = src[i * cstride:i * cstride + z]
        l.libdeflate_b200_pinned_free(tmp)

    def e2e_step():
        if args.workload == "roundtrip":
            ctx._check(l.libdeflate_b200_compress_batch_host_packed(ctx.h, fmt, LEVEL, in_ptrs.ctypes.data, in_sizes.ctypes.data, ne,
                                                                    pin_comp, packed_cap, comp_offs.ctypes.data, comp_sizes.ctypes.data), "compress_batch_host_packed")
        ctx._check(l.libdeflate_b200_decompress_batch_host_packed(ctx.h, fmt, 0, pin_comp, comp_offs.ctypes.data, comp_sizes.ctypes.data, ne,
                                                                  out_ptrs.ctypes.data, out_avail.ctypes.data, None, aout.ctypes.data, res.ctypes.data), "decompress_batch_host_packed")
    host_in = np.ctypeslib.as_array(ctypes.cast(pin_in, ctypes.POINTER(ctypes.c_uint8)), shape=(ne * chunk,))
    host_out = np.ctypeslib.as_array(ctypes.cast(pin_out, ctypes.POINTER(ctypes.c_uint8)), shape=(ne * chunk,))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    ksteps = max(1, min(args.steps, 3))

    def measure(step):
        for _ in range(min(args.warmup, 2)):
            step()
        res[:] = -1
        aout[:] = 0
        host_out[:4096] = 0
        barrier()
        t0 = time.perf_counter()
        for _ in range(ksteps):
            step()
        dt = allmax(time.perf_counter() - t0)
        assert (res == 0).all() and (aout == chunk).all()
        assert np.array_equal(host_in, host_out), "e2e round trip mismatch"
        return world * ne * chunk * ksteps / 1e6 / dt

    val = measure(e2e_step)
    comp_total = int(comp_sizes.sum())
    packed_total = int(comp_offs[ne])
    mode = "one host thread: compress call, then decompress call, whole batch each"
    serial_val, groups, two_thread_val = val, 0, None
    if args.workload == "roundtrip" and ne >= int(os.environ.get("LDB_E2E_GROUP_MIN", "4096")) and getattr(args, "overlap", False):
        # The same two calls with the batch going through in GROUPS: one host thread compresses group g + 1 (own
        # context = own stream) while a second one decompresses group g, to hide the decompress call's PCIe time
        # behind the deflate kernel of the next group.  Measured: it does not pay (profiles/r02_e2e_overlap.md).
        import threading
        groups = 4
        ng = ne // groups
        ctx2 = ldb.Context(ctx.device, l)
        gcap = ng * (cstride + 16)
        g_offs = [np.zeros(ng + 1, dtype=np.uint64) for _ in range(groups)]
        g_sizes = [np.zeros(ng, dtype=np.uint64) for _ in range(groups)]

        trace = [] if os.environ.get("LDB_E2E_TRACE") else None

        def overlapped_step():
            done = [threading.Event() for _ in range(groups)]
            err = []
            t_base = time.perf_counter()
            if trace is not None:
                trace.clear()

            def comp():
                try:
                    for g in range(groups):
                        lo = g * ng
                        ctx._check(l.libdeflate_b200_compress_batch_host_packed(ctx.h, fmt, LEVEL, in_ptrs[lo:].ctypes.data, in_sizes[lo:].ctypes.data, ng,
                                                                                pin_comp + g * gcap, gcap, g_offs[g].ctypes.data, g_sizes[g].ctypes.data), "compress_batch_host_packed")
                        if trace is not None:
                            trace.append(("compress %d done" % g, round(1e3 * (time.perf_counter() - t_base), 1)))
                        done[g].set()
                except Exception as e:      # noqa: BLE001
                    err.append(e)
                    for d in done:
                        d.set()
            t = threading.Thread(target=comp)
            t.start()
            for g in range(groups):
                done[g].wait()
                if err:
                    break
                lo = g * ng
                ctx2._check(l.libdeflate_b200_decompress_batch_host_packed(ctx2.h, fmt, 0, pin_comp + g * gcap, g_offs[g].ctypes.data, g_sizes[g].ctypes.data, ng,
                                                                           out_ptrs[lo:].ctypes.data, out_avail[lo:].ctypes.data, None, aout[lo:].ctypes.data, res[lo:].ctypes.data),
                            "decompress_batch_host_packed")
                if trace is not None:
                    trace.append(("decompress %d done" % g, round(1e3 * (time.perf_counter() - t_base), 1)))
            t.join()
            if err:
                raise err[0]
        if ng * groups == ne:
            oval = measure(overlapped_step)
            assert sum(int(z.sum()) for z in g_sizes) == comp_total      # the same streams as the one-call form
            two_thread_val = oval
            if trace:
                print("e2e two-thread timeline of the last step (ms):", sorted(trace, key=lambda t: t[1]), file=sys.stderr)
            if oval > val:
                val = oval
                mode = "two host threads, %d groups of %d chunks: compressing group g+1 overlaps decompressing group g" % (groups, ng)
        ctx2.close()
    small = 16 * ne + 8 * (ne + 1)      # size / offset tables
    if args.workload == "roundtrip":
        h2d = ne * chunk + packed_total + small
        d2h = packed_total + ne * chunk + small
    else:
        h2d = packed_total + small
        d2h = ne * chunk + small
    l.libdeflate_b200_pinned_free(pin_comp)
    l.libdeflate_b200_pinned_free(pin_out)
    return {"value": round(val, 2), "unit": "MB/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
            "payload_compressed_bytes": comp_total, "packed_compressed_bytes": packed_total, "chunks_per_gpu": ne, "steps": ksteps,
            "mode": mode, "one_thread_value": round(serial_val, 2), "two_thread_value": None if two_thread_val is None else round(two_thread_val, 2),
            "api": "libdeflate_b200_compress_batch_host_packed + libdeflate_b200_decompress_batch_host_packed" if args.workload == "roundtrip"
                   else "libdeflate_b200_decompress_batch_host_packed",
            "timing": "host wall clock around the synchronous host calls, max over ranks"}


def main():
    global LEVEL
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="roundtrip", choices=["roundtrip", "decompress"])
    ap.add_argument("--chunks", type=int, default=NCHUNKS_DEFAULT)
    ap.add_argument("--chunk-size", type=int, default=CHUNK_DEFAULT)
    ap.add_argument("--level", type=int, default=LEVEL, help="compression level (BASELINE configs[3] uses 12 with --chunk-size 1048576 --chunks 4096)")
    ap.add_argument("--data-class", type=int, default=0, help="synthetic chunk class (bench/synth.c): 0 text (the headline corpus), 1 pattern, 2 stride, 3 random, 4 zeros, 5 mixed, 6 all of them in turn")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the short legs of the other BASELINE configs (decompress-only, checksums, level 12)")
    ap.add_argument("--no-l12", action="store_true", help="skip the level-12 4096 x 1 MiB leg")
    ap.add_argument("--overlap", action="store_true", help="e2e: also measure the two-host-thread form (compress of group g+1 over decompress of group g); "
                    "measured slower than the plain form (9.3 vs 10.06 GB/s, profiles/r02_e2e_overlap.md), hence off by default")
    ap.add_argument("--no-origin", action="store_true", help="N > 1: skip the single-origin (NCCL scatter/gather) leg")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed (rank 0's shard) to DIR/<name>.npy")
    args = ap.parse_args()
    LEVEL = args.level
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
