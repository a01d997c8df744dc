"""Regenerates the committed golden fixtures.  Needs /root/reference (it runs the
UNMODIFIED reference built into oracle/_ref/); the fixtures themselves travel with the repo.

    python tests/golden/make_fixtures.py [ref_streams] [known_answers] [reference_answers]

ref_streams.npz   : streams produced by the reference COMPRESSOR (levels 1/6/9/12, three
                    formats) with their plain texts -> pins bit-exact decompression.
known_answer.json : hand-assembled raw-DEFLATE streams in the spirit of the reference's
                    programs/test_incomplete_codes.c, test_invalid_streams.c, test_overread.c
                    and test_slow_decompression.c, with the verdict and output bytes the
                    reference returned for them here.
reference_answers.npz: the reference's answers for the inputs the tests compare with it
                    (tests/reference_answers.py builds those inputs and reads the answers back).
"""
import json
import os
import random
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import corpus  # noqa: E402
import deflate_asm as da  # noqa: E402
import parity_checks as pc  # noqa: E402
import reference_answers as ra  # noqa: E402
import libdeflate_b200 as ldb  # noqa: E402
from conftest import _load_ref  # noqa: E402

ref = ldb.Api(_load_ref(os.path.join(ROOT, "oracle", "_ref", "libdeflate_ref.so")))


def ref_streams():
    arrs = {}
    k = 0
    for n in (0, 1, 77, 4000, 65536):
        for name, plain in corpus.all_classes(n, 1000 + n).items():
            if n == 65536 and name not in ("T", "M"):
                continue
            for fmt in (0, 1, 2):
                for lvl in (1, 6, 9, 12):
                    if n == 65536 and lvl in (9,):
                        continue
                    z = ref.compress(plain, lvl, fmt)
                    key = "f%d_%s_%d_L%d_%d" % (fmt, name, n, lvl, k)
                    arrs[key + "_p"] = np.frombuffer(plain, dtype=np.uint8)
                    arrs[key + "_z"] = np.frombuffer(z, dtype=np.uint8)
                    k += 1
    np.savez_compressed(os.path.join(HERE, "ref_streams.npz"), **arrs)
    print("ref_streams.npz:", k, "streams")


def known_answers():
    cases = []

    def add(name, stream, out_avail):
        r = ref.decompress(stream, out_avail, 0)
        cases.append({"name": name, "stream": stream.hex(), "out_avail": out_avail, "result": r[0],
                      "output": r[1].hex() if r[0] == 0 else ""})

    # (1) empty offset code, literals only  (cf. test_incomplete_codes.c:73 "ABAA")
    ll = [0] * 288
    ll[ord("A")] = 1
    ll[ord("B")] = 2
    ll[256] = 2
    bw = da.BitWriter()
    da.dynamic_block(bw, ll, [0] * 32, [65, 66, 65, 65])
    add("empty_offset_code", bw.bytes(), 128)
    # (2) litlen code with a single symbol (EOB, length 1)  (cf. :155)
    ll = [0] * 288
    ll[256] = 1
    bw = da.BitWriter()
    da.dynamic_block(bw, ll, [0] * 32, [])
    add("singleton_litlen_code", bw.bytes(), 128)
    # (3) offset code with the single symbol 0  (cf. :215, expected 255 x4)
    ll = [0] * 288
    ll[255] = 1
    ll[256] = 2
    ll[257] = 2
    ol = [0] * 32
    ol[0] = 1
    bw = da.BitWriter()
    da.dynamic_block(bw, ll, ol, [255, (3, 1)])
    add("singleton_offset_code_sym0", bw.bytes(), 128)
    # (4) offset code with a single non-zero symbol  (cf. :292, expected 254 255 254 255 254)
    ol = [0] * 32
    ol[1] = 1
    ll = [0] * 288
    ll[254] = 2
    ll[255] = 2
    ll[256] = 2
    ll[257] = 2
    bw = da.BitWriter()
    da.dynamic_block(bw, ll, ol, [254, 255, (3, 2)])
    add("singleton_offset_code_sym1", bw.bytes(), 128)
    # (5) singleton code of length 2 is NOT accepted (incomplete)
    ll = [0] * 288
    ll[256] = 2
    bw = da.BitWriter()
    da.dynamic_block(bw, ll, [0] * 32, [])
    add("incomplete_litlen_len2", bw.bytes(), 128)
    # (6) overfull litlen code
    ll = [0] * 288
    ll[65] = 1
    ll[66] = 1
    ll[256] = 1
    bw = da.BitWriter()
    da.dynamic_block(bw, ll, [0] * 32, [65])
    add("overfull_litlen_code", bw.bytes(), 128)
    # (7) too many codeword lengths (cf. test_invalid_streams.c:59): zero-run past the end
    bw = da.BitWriter()
    bw.put(1, 1); bw.put(2, 2); bw.put(0, 5); bw.put(0, 5); bw.put(15, 4)
    for s in da.PERM:
        bw.put(da.PRECODE_LENS[s], 3)
    pc = da.canonical(da.PRECODE_LENS)
    for _ in range(2):
        bw.put_code(pc[18], da.PRECODE_LENS[18]); bw.put(127, 7)      # 138 + 138 > 258
    add("too_many_codeword_lengths", bw.bytes(), 128)
    # (8) stream that runs off its end into implicit zeros (cf. test_overread.c:71-95):
    #     must be BAD_DATA, not INSUFFICIENT_SPACE, even with plenty of output space
    ll = [0] * 288
    ll[0] = 1
    ll[256] = 1
    bw = da.BitWriter()
    da.dynamic_block(bw, ll, [0] * 32, [0] * 5, emit_eob=False)
    add("overread_into_zeros_big_out", bw.bytes(), 100000)
    add("overread_into_zeros_small_out", bw.bytes(), 7)
    # (9) stored blocks: good, bad NLEN, truncated
    add("stored_ok", bytes([1, 3, 0, 0xfc, 0xff, 9, 8, 7]), 16)
    add("stored_bad_nlen", bytes([1, 3, 0, 0xfc, 0xfe, 9, 8, 7]), 16)
    add("stored_truncated", bytes([1, 3, 0, 0xfc, 0xff, 9, 8]), 16)
    add("stored_no_room", bytes([1, 3, 0, 0xfc, 0xff, 9, 8, 7]), 2)
    # (10) reserved block type
    add("btype_3", bytes([7, 0, 0, 0, 0]), 16)
    # (11) match reaching before the start of the output
    ll = [0] * 288
    ll[65] = 2; ll[256] = 2; ll[257] = 1
    ol = [0] * 32
    ol[2] = 1; ol[3] = 1
    bw = da.BitWriter()
    da.dynamic_block(bw, ll, ol, [65, (3, 3)])
    add("offset_too_far", bw.bytes(), 128)
    # (12) floods of empty blocks (cf. test_slow_decompression.c:427-472), small versions
    bw = da.BitWriter()
    for i in range(200):
        bw.put(0, 1); bw.put(1, 2); bw.put(0, 7)           # empty static block
    bw.put(1, 1); bw.put(1, 2); bw.put(0, 7)
    add("empty_static_blocks", bw.bytes(), 16)
    # (13) long codewords / many subtables (decoder table overflow path)
    rng = random.Random(99)
    for i in range(6):
        z, p = da.odd_code_stream(rng, n_tokens=600)
        add("odd_complete_codes_%d" % i, z, len(p))
        add("odd_complete_codes_%d_short_out" % i, z, len(p) - 1)
    # (14) litlen symbols 286/287 and offset symbols 30/31 are accepted by the reference
    ll = [0] * 288
    ll[65] = 2; ll[256] = 2; ll[286] = 2; ll[287] = 2
    ol = [0] * 32
    ol[0] = 1; ol[30] = 1
    bw = da.BitWriter()
    lc, oc = da.canonical(ll), da.canonical(ol)
    bw.put(1, 1); bw.put(2, 2); bw.put(288 - 257, 5); bw.put(31 - 1, 5); bw.put(15, 4)
    for s in da.PERM:
        bw.put(da.PRECODE_LENS[s], 3)
    da.write_code_lengths(bw, ll[:288] + ol[:31])
    bw.put_code(lc[65], 2)
    bw.put_code(lc[286], 2); bw.put_code(oc[0], 1)          # length 258, offset 1
    bw.put_code(lc[287], 2); bw.put_code(oc[0], 1)
    bw.put_code(lc[256], 2)
    add("litlen_286_287", bw.bytes(), 1000)
    with open(os.path.join(HERE, "known_answer.json"), "w") as f:
        json.dump(cases, f, indent=0)
    for c in cases:
        print("%-40s result=%d out=%d bytes" % (c["name"], c["result"], len(c["output"]) // 2))


def reference_answers():
    arrs = {}

    def record(name, cases, answer):
        arrs[name] = np.array([answer(c) for c in cases], dtype=np.uint64)
        arrs[name + "_inputs"] = np.array(ra.inputs_digest(cases))

    record("checksums", ra.checksum_cases(), lambda c: (ref.crc32(c[0], c[1]), ref.adler32(c[0], c[2])))
    record("valid_streams", ra.valid_stream_cases(), lambda c: ra.outcome(ref.decompress(c[2], len(c[1]), c[0])))
    record("fuzz", ra.fuzz_cases(), lambda c: ra.outcome(ref.decompress(c[1], c[2], c[0], c[3])))
    record("gzip_header", pc.gzip_header_cases(), lambda c: ra.outcome(ref.decompress(c[1], len(c[0]), 2)))
    names = ("deflate", "zlib", "gzip")
    record("bound_and_stored", [(n, fmt) for n in ra.STORED_SIZES for fmt in (0, 1, 2)],
           lambda c: (getattr(ref.l, "libdeflate_%s_compress_bound" % names[c[1]])(None, c[0]),
                      ra.digest(ref.compress(corpus.rand(c[0], c[0]), 0, c[1]))))
    chunks = ra.emu_deflate_chunks()
    for name, levels, fmt in ra.EMU_DEFLATE_RUNS:
        record("emu_deflate_" + name, chunks, lambda c: [len(ref.compress(c, lvl, fmt)) for lvl in levels])
    record("levels_10_12", ra.chunks_1mib(), lambda c: [len(ref.compress(c, lvl, 0)) for lvl in ra.LEVELS_10_12])
    import bench
    for i, p in zip(ra.FULL_SIZE_INDICES, ra.full_size_plains(bench.load_synth())):
        arrs["full_size_gzip6_%d" % i] = np.frombuffer(ref.compress(p, 6, 2), dtype=np.uint8)
    np.savez_compressed(os.path.join(HERE, "reference_answers.npz"), **arrs)
    print("reference_answers.npz:", {k: v.shape for k, v in arrs.items()})


if __name__ == "__main__":
    for step in sys.argv[1:] or ["ref_streams", "known_answers", "reference_answers"]:
        globals()[step]()
