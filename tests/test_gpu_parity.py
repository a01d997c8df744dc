"""`-m gpu`: the parity tests proper -- CUDA path (through the C ABI) vs the oracle, zlib
and the reference-built fixtures, on a real B200."""
import ctypes
import glob
import os
import subprocess
import sys
import zlib

import numpy as np
import pytest

import corpus
import parity_checks as pc
import reference_answers as ra

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
pytestmark = pytest.mark.gpu


NATIVE_ONLY = """
import libdeflate_b200 as ldb
assert ldb.lib().libdeflate_b200_device_count() >= 1
maps = open("/proc/self/maps").read()
assert "libdeflate_b200.so" in maps and "libdeflate_b200_emu" not in maps
"""


def test_native_library_is_loaded():
    import libdeflate_b200 as ldb
    assert ldb.lib().libdeflate_b200_device_count() >= 1
    assert ldb.lib()._name == ldb.LIB_PATH and os.path.basename(ldb.LIB_PATH) == "libdeflate_b200.so"
    assert "libdeflate_b200.so" in open("/proc/self/maps").read()
    # the package on its own loads the nvcc build and never the emulator build; checked in a fresh
    # interpreter, since the CPU tests of the same session load the emulator build into this one
    r = subprocess.run([sys.executable] + (["-s"] if sys.flags.no_user_site else []) + ["-c", NATIVE_ONLY], cwd=ROOT,
                       stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=300)
    assert r.returncode == 0, r.stdout.decode()[-2000:]


def test_checksums_single_call(gpu_api, oracle):
    pc.check_checksums(gpu_api, oracle)


def test_checksums_batch(gpu_ctx, oracle):
    pc.check_checksum_batch(gpu_ctx, oracle, n_chunks=300, max_len=300000)


def test_checksums_every_alignment(gpu_ctx):
    """ref: programs/test_checksums.c:154-200 -- every start alignment, ragged lengths."""
    rng = np.random.default_rng(5)
    blob = rng.integers(0, 256, 70000, dtype=np.uint8).tobytes()
    bufs = [blob[a:a + ln] for a in range(0, 33) for ln in (0, 1, 31, 32, 33, 1000, 32768 + a)]
    assert gpu_ctx.checksum_batch_host(bufs, "crc32") == [zlib.crc32(b) for b in bufs]
    assert gpu_ctx.checksum_batch_host(bufs, "adler32") == [zlib.adler32(b) for b in bufs]


def test_decompress_valid_streams(gpu_ctx, oracle):
    streams = pc.make_valid_streams(sizes=(0, 1, 100, 5000, 65536), levels=(1, 6, 9))
    pc.check_decompress_valid(gpu_ctx, oracle, streams)


def test_decompress_reference_fixture_streams(gpu_ctx, oracle):
    """Streams produced by the UNMODIFIED reference compressor (committed fixtures)."""
    fx = np.load(os.path.join(ROOT, "tests", "golden", "ref_streams.npz"))
    names = sorted(k[:-2] for k in fx.files if k.endswith("_z"))
    for fmt in (0, 1, 2):
        sel = [n for n in names if n.startswith("f%d_" % fmt)]
        plains = [fx[n + "_p"].tobytes() for n in sel]
        zs = [fx[n + "_z"].tobytes() for n in sel]
        got = gpu_ctx.decompress_batch_host(zs, [len(p) for p in plains], fmt)
        for g, p, z in zip(got, plains, zs):
            assert g[0] == 0 and g[1] == p and g[2] == len(z)


def test_decompress_1mib_chunks(gpu_ctx, oracle):
    plains = [corpus.text(1 << 20, 3), corpus.mixed(1 << 20, 4), corpus.zeros(1 << 20)]
    zs = [corpus.zlib_raw(p, 9) for p in plains]
    got = gpu_ctx.decompress_batch_host(zs, [len(p) for p in plains], 0)
    for g, p in zip(got, plains):
        assert g[0] == 0 and g[1] == p


def test_packed_host_forms(gpu_ctx):
    pc.check_packed_round_trip(gpu_ctx, n_chunks=3000, fmts=(0, 1, 2))


def test_host_inputs_with_unmapped_gaps(gpu_ctx):
    pc.check_inputs_with_unmapped_gaps(gpu_ctx)


def test_gzip_optional_header_fields(gpu_ctx, oracle):
    pc.check_gzip_optional_fields(gpu_ctx, oracle)


def test_compress_1mib_chunks_levels_10_12(gpu_ctx, oracle):
    """BASELINE configs[3] shape: 1 MiB chunks through the near-optimal levels (the ring is crossed 16 times, the
    DP segment logic 512 times per chunk): round trip, bound, and the ratio next to the reference's."""
    chunks = ra.chunks_1mib()
    ref_sizes = ra.answers("levels_10_12", chunks)
    for k, lvl in enumerate(ra.LEVELS_10_12):
        zs = gpu_ctx.compress_batch_host(chunks, lvl, 0)
        for c, z, rs in zip(chunks, zs, ref_sizes):
            assert z is not None and len(z) <= oracle.l.oracle_compress_bound(0, len(c))
            assert zlib.decompress(z, -15) == c
            r = oracle.decompress(z, len(c), 0)
            assert r[0] == 0 and r[1] == c and r[2] == len(z)
            # (measured: 13 % behind at level 10 on this very repetitive text -- no length-3 matches, 2 cost passes;
            # the guard is a regression fence, the numbers are in DESIGN.md)
            # + 1 KiB: our blocks end every 32 KiB, 32 block headers per MiB show on inputs that shrink to ~1 KB (zeros: 1838 vs 1070 B)
            assert len(z) <= 1.16 * rs[k] + 1024, ("ratio vs reference", lvl, len(z), rs[k])


def test_two_contexts_two_host_threads(gpu_ctx):
    """Distinct objects may be used concurrently from different threads (ref: libdeflate.h:56-57, 178-179): two
    contexts, two threads, plus the classic single-buffer API from both at once."""
    import threading
    import libdeflate_b200 as ldb
    errs = []

    def work(seed):
        try:
            ctx = ldb.Context(0)
            api = ldb.Api()
            chunks = [corpus.text(30000 + 17 * i, seed * 100 + i) for i in range(40)]
            for _ in range(3):
                zs = ctx.compress_batch_host(chunks, 6, 2)
                got = ctx.decompress_batch_host(zs, [len(c) for c in chunks], 2)
                assert all(g[0] == 0 and g[1] == c for g, c in zip(got, chunks))
                z = api.compress(chunks[0], 6, 1)
                assert api.decompress(z, len(chunks[0]), 1)[1] == chunks[0]
        except Exception as e:      # noqa: BLE001
            errs.append(repr(e))
    ts = [threading.Thread(target=work, args=(s,)) for s in (1, 2)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errs, errs


def test_two_devices_one_process():
    """Kernel attributes are per device: a second context on another GPU of the same process must work."""
    import libdeflate_b200 as ldb
    if ldb.lib().libdeflate_b200_device_count() < 2:
        pytest.skip("needs 2 GPUs (run through gpurun --gpus 2)")
    chunks = [corpus.text(65536, i) for i in range(64)]
    outs = []
    for dev in (0, 1, 0):
        ctx = ldb.Context(dev)
        zs = ctx.compress_batch_host(chunks, 6, 2)
        got = ctx.decompress_batch_host(zs, [len(c) for c in chunks], 2)
        assert all(g[0] == 0 and g[1] == c for g, c in zip(got, chunks))
        outs.append(zs)
    assert outs[0] == outs[1] == outs[2]


def test_decompress_token_scratch_waves(gpu_ctx, oracle):
    pc.check_decompress_in_waves(gpu_ctx, oracle, n_chunks=400)


def test_decompress_large_chunks(gpu_ctx):
    pc.check_decompress_large(gpu_ctx)


def test_decompress_fuzz_verdicts(gpu_ctx, oracle):
    seen = pc.check_decompress_fuzz(gpu_ctx, oracle, pc.fuzz_cases(6000, seed=77))
    assert set(seen) == {0, 1, 2, 3}, seen


def test_decompress_truncation_and_space_sweep(gpu_ctx, oracle):
    """Every cut of the last 48 input bytes and every output size around the exact one (multi-symbol decode step)."""
    pc.check_truncation_and_space_sweep(gpu_ctx, oracle)


def test_known_answer_fixtures(gpu_ctx, oracle):
    """ref: programs/test_incomplete_codes.c, test_invalid_streams.c, test_overread.c --
    hand-assembled streams with expected bytes / verdicts (tests/golden/known_answer.json)."""
    import json
    ka = json.load(open(os.path.join(ROOT, "tests", "golden", "known_answer.json")))
    zs = [bytes.fromhex(k["stream"]) for k in ka]
    got = gpu_ctx.decompress_batch_host(zs, [k["out_avail"] for k in ka], 0)
    for k, g in zip(ka, got):
        assert g[0] == k["result"], k["name"]
        if k["result"] == 0:
            assert g[1] == bytes.fromhex(k["output"]), k["name"]


def test_single_buffer_api_round_trip(gpu_api, oracle):
    for n in (0, 1, 54, 55, 56, 1000, 65536, 200000):
        d = corpus.text(n, n)
        for fmt in (0, 1, 2):
            for lvl in (0, 1, 6, 9, 12):
                z = gpu_api.compress(d, lvl, fmt)
                assert z is not None
                assert len(z) <= oracle.l.oracle_compress_bound(fmt, n)
                r = oracle.decompress(z, n, fmt)
                assert r[0] == 0 and r[1] == d
                wb = {0: -15, 1: 15, 2: 31}[fmt]
                assert zlib.decompress(z, wb) == d
                g = gpu_api.decompress(z, n, fmt)
                assert g[0] == 0 and g[1] == d and g[2] == len(z)
            # output too small => 0 (ref: libdeflate.h:85-88)
            if n:
                assert gpu_api.compress(d, 6, fmt, out_avail=4) is None


def test_compress_batch_round_trip_and_bound(gpu_ctx, oracle):
    chunks = []
    for n in (0, 1, 300, 5000, 65536):
        chunks += list(corpus.all_classes(n, n + 9).values())
    for fmt in (0, 1, 2):
        for lvl in (0, 1, 6, 9, 12):
            zs = gpu_ctx.compress_batch_host(chunks, lvl, fmt)
            for c, z in zip(chunks, zs):
                assert z is not None and len(z) <= oracle.l.oracle_compress_bound(fmt, len(c))
                r = oracle.decompress(z, len(c), fmt)
                assert r[0] == 0 and r[1] == c, (fmt, lvl, len(c))


def test_compress_stored_blocks_next_to_crossing_matches(gpu_ctx):
    pc.check_boundary_round_trip(gpu_ctx, levels=(1, 4, 6, 9, 10, 12), fmt=2)


def test_compress_random_mix(gpu_ctx):
    pc.check_random_mix_round_trip(gpu_ctx, seed=7, rounds=12, per_round=24)


def test_bgzf(gpu_ctx):
    pc.check_bgzf(gpu_ctx, sizes=(0, 1, 65279, 65280, 65281, 200000, 3000000), levels=(1, 6, 9))


def test_gz_front_end(gpu_ctx, gpu_api, tmp_path):
    """python -m libdeflate_b200.gz (gzip-style front end, SURVEY section 8 row f1) on the GPU: what it writes is read by
    Python's gzip, what it reads back is identical, blocked and plain multi-member files both decode."""
    import gzip
    import corpus
    from libdeflate_b200 import gz
    data = corpus.text(3000000, 9) + corpus.rand(70000, 9) + corpus.zeros(100000)
    f = tmp_path / "a.bin"
    f.write_bytes(data)
    assert gz.main(["-6", "-k", str(f)], ctx=gpu_ctx) == 0
    packed = (tmp_path / "a.bin.gz").read_bytes()
    assert gzip.decompress(packed) == data and gz.uncompressed_size(packed) == len(data)
    f.unlink()
    assert gz.main(["-d", str(tmp_path / "a.bin.gz")], ctx=gpu_ctx) == 0
    assert f.read_bytes() == data
    assert gz.decompress_bytes(gpu_ctx, pc.bgzf_reference_file(data)) == data
    plain = gzip.compress(data[:700000], 6) + gzip.compress(b"") + gzip.compress(data[700000:], 1)
    assert gz.decompress_members(gpu_api, plain) == data


def test_pipelined_host_path(gpu_ctx):
    import libdeflate_b200 as ldb
    pc.check_host_pipeline(ldb.lib(), gpu_ctx, n=8192, chunk=65536)


def test_full_size_property_round_trip(gpu_ctx):
    """BASELINE-sized batch: 4096 x 64 KiB chunks of the robustness mix T/P/S/R/Z/M, the reference's
    level-6 gzip streams in (the committed streams of 21 distinct chunks, cycled through the batch),
    checksum-of-checksums out (size-independent property)."""
    import bench
    plains = ra.full_size_plains(bench.load_synth())
    fx = ra.load()
    streams = [fx["full_size_gzip6_%d" % i].tobytes() for i in ra.FULL_SIZE_INDICES]
    n, chunk = 4096, ra.FULL_SIZE_CHUNK
    got = gpu_ctx.decompress_batch_host([streams[i % len(streams)] for i in range(n)], chunk, 2)
    crcs = [zlib.crc32(p) for p in plains]
    for i, g in enumerate(got):
        assert g[0] == 0 and g[3] == chunk
        assert zlib.crc32(g[1]) == crcs[i % len(crcs)]


def test_reference_test_programs_against_our_library():
    """Drop-in acceptance: the reference's own programs/test_*.c, compiled UNMODIFIED here
    against libdeflate_b200.so (oracle/Makefile `reftests`), run on the GPU box."""
    progs = sorted(glob.glob(os.path.join(ROOT, "oracle", "_ref", "test_*")))
    if not progs:
        pytest.skip("oracle/_ref/test_* not prebuilt")
    for p in progs:
        if os.path.basename(p) == "test_slow_decompression":
            continue        # opt-in perf test in the reference as well (INCLUDE_PERF_TESTS)
        r = subprocess.run([p], stdout=subprocess.PIPE, stderr=subprocess.STDOUT, timeout=600)
        assert r.returncode == 0, (p, r.stdout.decode()[-2000:])


def _nccl_origin_worker(rank, world, port, n_total, chunk, q):
    import torch
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    import libdeflate_b200 as ldb
    from libdeflate_b200 import shard
    import bench
    ctx = ldb.Context(rank)
    dev = torch.device("cuda", rank)
    rt = shard.OriginRoundTrip(ctx, dist, dev, n_total, chunk, ldb.GZIP, 6, stages=4)
    root_in = None
    if rank == 0:
        synth = bench.load_synth()
        buf = (ctypes.c_uint8 * (n_total * chunk))()
        synth.synth_fill(buf, chunk, 0, n_total, 0, 4)
        root_in = torch.frombuffer(bytearray(bytes(buf)), dtype=torch.uint8).to(dev)
    for _ in range(2):
        info = rt.step(root_in)
    ok = bool((rt.res[:rt.n] == 0).all().item())
    if rank == 0:
        raw = bytes(root_in.cpu().numpy())
        ok = ok and bytes(rt.out_all.cpu().numpy()) == raw
        offs, sizes, comp = rt.comp_offsets.tolist(), rt.comp_sizes.tolist(), bytes(rt.comp_all.cpu().numpy())
        for i in range(0, n_total, 97):
            ok = ok and zlib.decompress(comp[offs[i]:offs[i] + sizes[i]], 31) == raw[i * chunk:(i + 1) * chunk]
        q.put((ok, info))
    dist.barrier()
    dist.destroy_process_group()


def test_two_gpu_single_origin_round_trip_over_nccl():
    """A real sharded batch through the NCCL scatter/gather data plane (needs two GPUs in the box)."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs (run through gpurun --gpus 2)")
    import torch.multiprocessing as mp
    world, n_total, chunk = 2, 4099, 65536
    mctx = mp.get_context("spawn")
    q = mctx.Queue()
    port = 33500 + os.getpid() % 2000
    procs = [mctx.Process(target=_nccl_origin_worker, args=(r, world, port, n_total, chunk, q)) for r in range(world)]
    for p in procs:
        p.start()
    ok, info = q.get(timeout=600)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    assert ok
    assert info["nvlink_bytes"]["root_out"] == (n_total - n_total // 2) * chunk
