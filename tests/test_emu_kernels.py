"""Kernel LOGIC on the CPU: the .cu sources compiled against tests/emu (SIMT emulator).

This is test infrastructure (the dev container has no GPU); the product path is only
ever the nvcc build, exercised by test_gpu_parity.py under `-m gpu`.
"""
import pytest
import parity_checks as pc
import reference_answers as ra


def test_checksum_kernels_emulated(emu_api, oracle):
    pc.check_checksums(emu_api, oracle, sizes=[0, 1, 15, 16, 17, 33, 511, 512, 513, 5553, 65536, 262144 + 17])


def test_checksum_batch_emulated(emu_ctx, oracle):
    pc.check_checksum_batch(emu_ctx, oracle, n_chunks=40, max_len=20000)


def test_inflate_valid_streams_emulated(emu_ctx, oracle):
    streams = pc.make_valid_streams(sizes=(0, 1, 100, 5000, 40000), levels=(1, 6)) + ra.fixture_streams()
    pc.check_decompress_valid(emu_ctx, oracle, streams)


def test_gzip_optional_header_fields_emulated(emu_ctx, oracle):
    pc.check_gzip_optional_fields(emu_ctx, oracle, ra.answers("gzip_header", pc.gzip_header_cases()))


def test_inflate_truncation_and_space_sweep_emulated(emu_ctx, oracle):
    pc.check_truncation_and_space_sweep(emu_ctx, oracle)


def test_inflate_token_scratch_waves_emulated(emu_ctx, oracle):
    pc.check_decompress_in_waves(emu_ctx, oracle, n_chunks=40)


def test_inflate_large_chunks_emulated(emu_ctx):
    pc.check_decompress_large(emu_ctx, sizes=(150000,), levels=(0, 6))


def test_inflate_fuzz_emulated(emu_ctx, oracle):
    v = pc.check_decompress_fuzz(emu_ctx, oracle, pc.fuzz_cases(1500, seed=11))
    assert set(v) >= {0, 1, 3}, v


def test_deflate_round_trip_emulated(emu_ctx, oracle):
    chunks = ra.emu_deflate_chunks()
    for name, levels, fmt in ra.EMU_DEFLATE_RUNS:
        ours = sum(pc.check_compress_round_trip(emu_ctx, oracle, chunks, levels=levels, fmts=(fmt,)))
        theirs = sum(sum(r) for r in ra.answers("emu_deflate_" + name, chunks))      # the reference's sizes
        assert ours <= theirs * 1.10, ("ratio regression", name, ours, theirs)
    pc.check_compress_round_trip(emu_ctx, oracle, chunks[:6], levels=(3, 9), fmts=(1,))


def test_deflate_stored_blocks_next_to_crossing_matches_emulated(emu_ctx):
    pc.check_boundary_round_trip(emu_ctx, levels=(1, 6), every=6)	# (the full sweep runs on the GPU)


def test_deflate_random_mix_emulated(emu_ctx):
    pc.check_random_mix_round_trip(emu_ctx, seed=3, rounds=3)


def test_bgzf_emulated(emu_ctx):
    pc.check_bgzf(emu_ctx, sizes=(0, 1, 65280, 65281, 140000), levels=(6,))


def test_gz_front_end_emulated(emu_ctx, emu_api, tmp_path):
    """The gzip-style front end (python -m libdeflate_b200.gz) on the emulated library: files written by it
    are read by Python's gzip, files it reads back are identical, -k / -c / level flags behave."""
    import gzip
    import corpus
    from libdeflate_b200 import gz
    data = corpus.text(150000, 9) + corpus.rand(5000, 9)
    f = tmp_path / "a.txt"
    f.write_bytes(data)
    assert gz.main(["-9", "-k", str(f)], ctx=emu_ctx) == 0
    packed = (tmp_path / "a.txt.gz").read_bytes()
    assert f.exists() and gzip.decompress(packed) == data and gz.uncompressed_size(packed) == len(data)
    f.unlink()
    assert gz.main(["-d", str(tmp_path / "a.txt.gz")], ctx=emu_ctx) == 0
    assert f.read_bytes() == data and not (tmp_path / "a.txt.gz").exists()
    assert gz.decompress_bytes(emu_ctx, pc.bgzf_reference_file(data)) == data
    with pytest.raises(ValueError):
        gz.decompress_bytes(emu_ctx, gzip.compress(data))
    # malformed size fields raise ValueError, never struct.error, and never drive a huge allocation
    import struct
    short_extra = bytes([0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 255]) + struct.pack("<H", 4000) + b"BC" + bytes(20)
    with pytest.raises(ValueError):
        gz.uncompressed_size(short_extra)
    liar = bytearray(packed[:-28])            # drop the EOF member, then lie in the last ISIZE
    liar[-4:] = struct.pack("<I", 0xFFFFFFF0)
    with pytest.raises(ValueError):
        gz.uncompressed_size(bytes(liar) * 1)
    # ordinary (not blocked) multi-member files go member by member through the classic API
    plain = gzip.compress(data[:70000], 6) + gzip.compress(b"") + gzip.compress(data[70000:], 1)
    assert gz.decompress_members(emu_api, plain) == data
    g = tmp_path / "b.gz"
    g.write_bytes(plain)
    assert gz.main(["-d", "-k", str(g)], ctx=emu_ctx, api=emu_api) == 0 and (tmp_path / "b").read_bytes() == data


def test_inflate_output_primitives_unit():
    """Randomized unit test of the resolve kernel's per-lane copy primitives (host build)."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "tests", "emu", "_build", "copy_unit")
    os.makedirs(os.path.dirname(exe), exist_ok=True)
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-DLDB_EMU", "-I", os.path.join(root, "tests", "emu"), "-include", "cuda_emu.h",
                           "-I", os.path.join(root, "libdeflate_b200", "csrc"), "-fno-strict-aliasing", "-Wno-unused-function", "-w",
                           os.path.join(root, "tests", "emu", "copy_unit.cpp"), os.path.join(root, "tests", "emu", "cuda_emu.cpp"),
                           "-o", exe, "-lpthread"])
    assert subprocess.run([exe]).returncode == 0


def test_packed_host_forms_emulated(emu_ctx):
    pc.check_packed_round_trip(emu_ctx, n_chunks=60)


def test_host_inputs_with_unmapped_gaps_emulated(emu_ctx):
    pc.check_inputs_with_unmapped_gaps(emu_ctx)


def test_pipelined_host_path_emulated(emu, emu_ctx):
    pc.check_host_pipeline(emu, emu_ctx)
