"""What the unmodified reference answered for the inputs the tests compare with it.

tests/golden/reference_answers.npz is written by tests/golden/make_fixtures.py, which runs the
reference; the tests only read it, so they need nothing outside the repository.  A decompress
answer is kept as (verdict, actual_in, actual_out, digest of the output bytes).  Every list of
answers is stored with a digest of the inputs it was recorded for, so inputs that come out
differently (another zlib, say) fail loudly instead of being compared with answers for other
inputs."""
import hashlib
import os
import random

import numpy as np

import corpus
import parity_checks as pc

HERE = os.path.dirname(os.path.abspath(__file__))
ANSWERS = os.path.join(HERE, "golden", "reference_answers.npz")
REF_STREAMS = os.path.join(HERE, "golden", "ref_streams.npz")

STORED_SIZES = (0, 1, 54, 55, 4999, 5000, 5001, 65535, 65536, 200000)
LEVELS_10_12 = (10, 12)
FULL_SIZE_CHUNK = 65536
# chunks of bench/synth.c class 6, the robustness mix (chunk i is of class i % 6: T P S R Z M).  P and Z chunks
# are the same at every index and S chunks repeat every 13 rounds (stride 1 + i % 13), so the first P and Z chunk
# and the S chunks of the first 13 rounds are every distinct one of them; T, M and R chunks all differ, and as
# their streams take 19 to 65 KB each, only the first three T, two M and one R chunk are kept
FULL_SIZE_INDICES = tuple(i for i in range(78) if i % 6 == 2 or (i % 6 == 0 and i < 18) or (i % 6 == 5 and i < 12) or i in (1, 3, 4))


def digest(data):
    """64-bit digest of a byte string (None, a failed call's output, is 0)."""
    if data is None:
        return 0
    return int.from_bytes(hashlib.blake2b(data, digest_size=8).digest(), "little")


def outcome(r):
    """(verdict, actual_in, actual_out, output digest) of a decompress call's (result, bytes, in, out)."""
    return (int(r[0]), int(r[2]), int(r[3]), digest(r[1]))


def inputs_digest(cases):
    h = hashlib.sha256()
    for case in cases:
        for f in (case if isinstance(case, tuple) else (case,)):
            b = f if isinstance(f, bytes) else str(f).encode()
            h.update(len(b).to_bytes(8, "little") + b)
    return h.hexdigest()


# ---- the inputs ----------------------------------------------------------------------------

def fixture_streams():
    """(format, plain, stream) of every stream the reference compressor made in ref_streams.npz."""
    fx = np.load(REF_STREAMS)
    names = sorted(k[:-2] for k in fx.files if k.endswith("_z"))
    return [(int(n[1]), fx[n + "_p"].tobytes(), fx[n + "_z"].tobytes()) for n in names]


def checksum_cases():
    """(data, crc32 initial value, adler32 initial value)"""
    rng = random.Random(1)
    out = []
    for n in pc.SIZES_CHECKSUM:
        d = rng.randbytes(n)
        for init in (0, 1, 0xCAFEBABE):
            out.append((d, init, init % ((65521 << 16)) if (init & 0xffff) < 65521 else 1))
    return out


def valid_stream_cases():
    """(format, plain, stream): zlib-made streams plus the reference compressor's own."""
    return pc.make_valid_streams(sizes=(0, 1, 100, 5000, 65536)) + fixture_streams()


def fuzz_cases():
    """(format, stream, out_avail, exact)"""
    return pc.fuzz_cases(6000, seed=2024)


def emu_deflate_chunks():
    return [b"", b"a", corpus.text(56, 1), corpus.text(3000, 2), corpus.pattern(9000), corpus.rand(6000, 3),
            corpus.zeros(70000), corpus.mixed(40000, 4), corpus.text(65536, 5), corpus.text(100000, 6)]


EMU_DEFLATE_RUNS = (("raw", (0, 1, 6, 12), 0), ("gzip", (6,), 2))      # (name, levels, format)


def chunks_1mib():
    return [corpus.text(1 << 20, 11), corpus.mixed(1 << 20, 12), corpus.rand(1 << 20, 13), corpus.zeros(1 << 20)]


def full_size_plains(synth):
    """The chunks FULL_SIZE_INDICES names, in that order."""
    import ctypes
    n = max(FULL_SIZE_INDICES) + 1
    buf = (ctypes.c_uint8 * (n * FULL_SIZE_CHUNK))()
    synth.synth_fill(buf, FULL_SIZE_CHUNK, 0, n, 6, 1)
    raw = bytes(buf)
    return [raw[i * FULL_SIZE_CHUNK:(i + 1) * FULL_SIZE_CHUNK] for i in FULL_SIZE_INDICES]


# ---- the answers ----------------------------------------------------------------------------

_answers = None


def load():
    global _answers
    if _answers is None:
        with np.load(ANSWERS) as f:
            _answers = {k: f[k] for k in f.files}
    return _answers


def answers(name, cases):
    """The reference's answers recorded under `name`, after checking they were recorded for `cases`."""
    a = load()
    assert str(a[name + "_inputs"]) == inputs_digest(cases), \
        "%s: the test inputs differ from those the reference answers were recorded for" % name
    return [tuple(int(x) for x in row) for row in a[name]]
