"""The deflate kernel's two schedules write the same streams (CPU, SIMT emulator).

Levels 1-9 run the search of pass s+1 on one warp group while another parses and encodes pass s;
-DLZ_PIPELINE=0 runs both halves on the whole CTA, one after the other.  Only the schedule differs,
so the compressed bytes must be identical, not merely close in size.
"""
import ctypes
import os
import subprocess

import pytest

import bench

CHUNK = 65536
NCHUNKS = 16


@pytest.fixture(scope="module")
def serial_ctx(emu, tmp_path_factory):
    """The emulator library with the deflate kernel built for the serial schedule."""
    import libdeflate_b200 as ldb
    from libdeflate_b200 import build as b
    out = str(tmp_path_factory.mktemp("serial_schedule"))
    objdir = os.path.dirname(b.EMU_LIB)
    cmd = ["g++", "-O1", "-std=c++17", "-fPIC", "-DLDB_EMU", "-DLZ_PIPELINE=0", "-I", b.EMU_DIR, "-include", "cuda_emu.h",
           "-Wno-unused-function", "-fno-strict-aliasing"]
    objs = []
    for src in b.SOURCES:
        if src == "deflate_kernel.cu":
            obj = os.path.join(out, "deflate_kernel.o")
            subprocess.check_call(cmd + ["-x", "c++", "-c", os.path.join(b.CSRC, src), "-o", obj])
        else:
            obj = os.path.join(objdir, src.replace(".cu", ".emu.o"))
        objs.append(obj)
    objs.append(os.path.join(objdir, "cuda_emu.o"))
    so = os.path.join(out, "libdeflate_b200_serial.so")
    subprocess.check_call(["g++", "-shared", "-o", so] + objs + ["-lpthread"])
    return ldb.Context(0, ldb.load_library(so))


def _chunks(data_class):
    synth = bench.load_synth()
    buf = (ctypes.c_uint8 * (NCHUNKS * CHUNK))()
    synth.synth_fill(buf, CHUNK, 0, NCHUNKS, data_class, 1)
    raw = bytes(buf)
    chunks = [raw[i * CHUNK:(i + 1) * CHUNK] for i in range(NCHUNKS)]
    # chunks that end inside the first, second and third quarter of the ring, and one below the stored-path size
    return chunks + [raw[:5000], raw[:16385], raw[:40000], raw[:30]]


@pytest.mark.parametrize("data_class", [0, 6], ids=["text", "robustness_mix"])
def test_pipelined_and_serial_schedules_write_identical_streams(emu_ctx, serial_ctx, data_class):
    import libdeflate_b200 as ldb
    chunks = _chunks(data_class)
    for level in range(1, 10):
        pipelined = emu_ctx.compress_batch_host(chunks, level=level, fmt=ldb.GZIP)
        serial = serial_ctx.compress_batch_host(chunks, level=level, fmt=ldb.GZIP)
        for i, (p, s) in enumerate(zip(pipelined, serial)):
            assert p == s, "level %d, chunk %d: %d vs %d bytes" % (level, i, len(p), len(s))
