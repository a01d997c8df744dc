"""pytest plumbing.

Markers:  gpu  -- needs a real B200 (run with `-m gpu` through gpurun).
Everything else runs on CPU: the oracle against golden vectors / the real reference,
the host logic, symbol export checks, and the kernel LOGIC through the SIMT emulator
(tests/emu, test infrastructure only -- never part of the product path).
"""
import ctypes
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run via gpurun")


def _have_gpu():
    try:
        import libdeflate_b200 as ldb
        return ldb.lib().libdeflate_b200_device_count() > 0
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    if _have_gpu():
        return
    skip = pytest.mark.skip(reason="no CUDA device here (GPU tests run through gpurun)")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


class Oracle:
    """ctypes view of oracle/liboracle.so (our C restatement; the checker)."""

    def __init__(self):
        d = os.path.join(ROOT, "oracle")
        so = os.path.join(d, "liboracle.so")
        srcs = [os.path.join(d, f) for f in ("inflate_oracle.c", "checksum_oracle.c", "oracle.h")]
        if not os.path.exists(so) or any(os.path.getmtime(s) > os.path.getmtime(so) for s in srcs):
            subprocess.check_call(["make", "-C", d, "liboracle.so"], stdout=subprocess.DEVNULL)
        self.l = ctypes.CDLL(so)
        self.l.oracle_crc32.restype = ctypes.c_uint32
        self.l.oracle_crc32.argtypes = [ctypes.c_uint32, ctypes.c_char_p, ctypes.c_size_t]
        self.l.oracle_adler32.restype = ctypes.c_uint32
        self.l.oracle_adler32.argtypes = [ctypes.c_uint32, ctypes.c_char_p, ctypes.c_size_t]
        self.l.oracle_decompress.restype = ctypes.c_int
        self.l.oracle_decompress.argtypes = [ctypes.c_int, ctypes.c_char_p, ctypes.c_size_t, ctypes.c_void_p,
                                             ctypes.c_size_t, ctypes.c_int, ctypes.POINTER(ctypes.c_size_t),
                                             ctypes.POINTER(ctypes.c_size_t)]
        self.l.oracle_compress_bound.restype = ctypes.c_size_t
        self.l.oracle_compress_bound.argtypes = [ctypes.c_int, ctypes.c_size_t]
        self.l.oracle_compress_stored.restype = ctypes.c_size_t
        self.l.oracle_compress_stored.argtypes = [ctypes.c_int, ctypes.c_int, ctypes.c_char_p, ctypes.c_size_t,
                                                  ctypes.c_void_p, ctypes.c_size_t]

    def crc32(self, data, crc=0):
        return self.l.oracle_crc32(crc, data, len(data))

    def adler32(self, data, adler=1):
        return self.l.oracle_adler32(adler, data, len(data))

    def decompress(self, data, out_avail, fmt=0, exact=False):
        out = ctypes.create_string_buffer(max(out_avail, 1))
        ain = ctypes.c_size_t(0)
        aout = ctypes.c_size_t(0)
        r = self.l.oracle_decompress(fmt, data, len(data), out, out_avail, 1 if exact else 0,
                                     ctypes.byref(ain), ctypes.byref(aout))
        if r != 0:
            return r, None, 0, 0
        n = out_avail if exact else aout.value
        return r, out.raw[:n], ain.value, n

    def compress_stored(self, data, fmt=0, level=0, out_avail=None):
        if out_avail is None:
            out_avail = self.l.oracle_compress_bound(fmt, len(data))
        out = ctypes.create_string_buffer(max(out_avail, 1))
        r = self.l.oracle_compress_stored(fmt, level, data, len(data), out, out_avail)
        return out.raw[:r] if r else None


@pytest.fixture(scope="session")
def oracle():
    return Oracle()


def _load_ref(so):
    """The UNMODIFIED reference (oracle/_ref/libdeflate_ref.so, for tests/golden/make_fixtures.py): it
    exports only the 21 classic symbols; attach just those prototypes."""
    import libdeflate_b200 as ldb
    lib = ctypes.CDLL(so)
    P, S, PS = ctypes.c_void_p, ctypes.c_size_t, ctypes.POINTER(ctypes.c_size_t)
    lib.libdeflate_alloc_compressor.restype = P
    lib.libdeflate_alloc_compressor.argtypes = [ctypes.c_int]
    lib.libdeflate_alloc_decompressor.restype = P
    lib.libdeflate_free_compressor.argtypes = [P]
    lib.libdeflate_free_compressor.restype = None
    lib.libdeflate_free_decompressor.argtypes = [P]
    lib.libdeflate_free_decompressor.restype = None
    for fmt in ("deflate", "zlib", "gzip"):
        f = getattr(lib, "libdeflate_%s_compress" % fmt)
        f.restype, f.argtypes = S, [P, P, S, P, S]
        f = getattr(lib, "libdeflate_%s_compress_bound" % fmt)
        f.restype, f.argtypes = S, [P, S]
        f = getattr(lib, "libdeflate_%s_decompress_ex" % fmt)
        f.restype, f.argtypes = ctypes.c_int, [P, P, S, P, S, PS, PS]
    lib.libdeflate_crc32.restype = ctypes.c_uint32
    lib.libdeflate_crc32.argtypes = [ctypes.c_uint32, P, S]
    lib.libdeflate_adler32.restype = ctypes.c_uint32
    lib.libdeflate_adler32.argtypes = [ctypes.c_uint32, P, S]
    return lib


@pytest.fixture(scope="session")
def emu():
    """The kernel sources compiled against the SIMT emulator (CPU, logic tests only)."""
    import libdeflate_b200 as ldb
    from libdeflate_b200 import build as b
    so = b.build_emu()
    return ldb.load_library(so)


@pytest.fixture(scope="session")
def emu_api(emu):
    import libdeflate_b200 as ldb
    return ldb.Api(emu)


@pytest.fixture(scope="session")
def emu_ctx(emu):
    import libdeflate_b200 as ldb
    return ldb.Context(0, emu)


@pytest.fixture(scope="session")
def gpu_ctx():
    import libdeflate_b200 as ldb
    return ldb.Context(0)


@pytest.fixture(scope="session")
def gpu_api():
    import libdeflate_b200 as ldb
    return ldb.Api()
