"""Parity checks shared by the emulator tests (CPU) and the GPU tests.

Every check drives the SAME C-ABI entry points (`api`/`ctx` wrap either the product
library on a B200 or the emulator build of the same kernel sources) and compares with
the oracle (`orc`), with zlib, and with what the unmodified reference answered for the same inputs
(tests/reference_answers.py).
"""
import random
import zlib

import corpus

SIZES_CHECKSUM = [0, 1, 2, 3, 15, 16, 17, 31, 32, 33, 63, 64, 255, 256, 511, 512, 513, 1024, 4095, 5552, 5553, 32768, 65536, 262144 + 17]


def check_checksums(api, orc, sizes=SIZES_CHECKSUM, seed=3):
    rng = random.Random(seed)
    for n in sizes:
        d = rng.randbytes(n)
        for init in (0, 0xDEADBEEF):
            assert api.crc32(d, init) == zlib.crc32(d, init) == orc.crc32(d, init), ("crc32", n, init)
        for init in (1, (65520 << 16) | 65520):
            assert api.adler32(d, init) == zlib.adler32(d, init) == orc.adler32(d, init), ("adler32", n, init)
    # NULL buffer -> initial values (ref: programs/test_checksums.c:63-71)
    assert api.crc32(None) == 0 and api.adler32(None) == 1
    # Adler-32 overflow vectors (ref: programs/test_checksums.c:176-196)
    d = b"\xff" * 5553
    init = (65520 << 16) | 65520
    assert api.adler32(d, init) == zlib.adler32(d, init)
    # multipart continuation (ref: programs/test_checksums.c:74-84)
    d = rng.randbytes(70000)
    for cut in (1, 100, 4097, 65535):
        assert api.crc32(d[cut:], api.crc32(d[:cut])) == zlib.crc32(d)
        assert api.adler32(d[cut:], api.adler32(d[:cut])) == zlib.adler32(d)


def check_checksum_batch(ctx, orc, n_chunks=67, max_len=70000, seed=4):
    rng = random.Random(seed)
    bufs = [rng.randbytes(rng.choice([0, 1, 15, 16, 17, 100, 4096, rng.randrange(max_len)])) for _ in range(n_chunks)]
    assert ctx.checksum_batch_host(bufs, "crc32") == [zlib.crc32(b) for b in bufs]
    assert ctx.checksum_batch_host(bufs, "adler32") == [zlib.adler32(b) for b in bufs]


def make_valid_streams(sizes=(0, 1, 100, 5000, 65536), levels=(1, 6, 9)):
    """(format, plain, stream) triples from zlib (independent producer); the reference compressor's own
    streams are reference_answers.fixture_streams() (SURVEY.md section 8c parity definition)."""
    out = []
    for n in sizes:
        for name, plain in corpus.all_classes(n, n + 5).items():
            for fmt, wb in ((0, -15), (1, 15), (2, 31)):
                for lv in levels:
                    out.append((fmt, plain, corpus.zlib_raw(plain, lv, zlib.Z_DEFAULT_STRATEGY, wb)))
                out.append((fmt, plain, corpus.zlib_raw(plain, 6, zlib.Z_FIXED, wb)))
                out.append((fmt, plain, corpus.zlib_raw(plain, 0, zlib.Z_DEFAULT_STRATEGY, wb)))
    return out


def check_decompress_valid(ctx, orc, streams):
    for fmt in (0, 1, 2):
        sel = [s for s in streams if s[0] == fmt]
        got = ctx.decompress_batch_host([s[2] for s in sel], [len(s[1]) for s in sel], fmt)
        for (f, plain, z), g in zip(sel, got):
            o = orc.decompress(z, len(plain), fmt)
            assert o[0] == 0 and o[1] == plain
            assert g == o, ("valid stream mismatch", fmt, len(plain), g[0], g[2:], o[2:])
        # exact-size mode and over-sized buffers
        got = ctx.decompress_batch_host([s[2] for s in sel], [len(s[1]) for s in sel], fmt, exact=True)
        assert all(g[0] == 0 and g[1] == s[1] for g, s in zip(got, sel))
        got = ctx.decompress_batch_host([s[2] for s in sel], [len(s[1]) + 77 for s in sel], fmt, exact=True)
        assert all(g[0] == (2 if True else 0) for g in got)	# SHORT_OUTPUT
        got = ctx.decompress_batch_host([s[2] for s in sel], [len(s[1]) + 77 for s in sel], fmt)
        assert all(g[0] == 0 and g[1] == s[1] for g, s in zip(got, sel))


def check_truncation_and_space_sweep(ctx, orc, n_text=6000):
    """The decode step takes several symbols at once (a match's length and offset, up to four literals behind
    a symbol).  What may NOT move with that: the over-read rule near the end of the input (evaluated per symbol
    start, ref: lib/deflate_decompress.c:236-254) and the "no room" verdicts.  So: one text stream cut at every
    byte of its last 48 bytes (plus a spread of earlier cuts), zero-extended, and every output size from a few
    bytes short to a few bytes long -- verdict, byte counts and bytes against the oracle."""
    plains = [corpus.text(n_text, 77), corpus.text(700, 78) + b"q" * 300 + corpus.text(500, 79), corpus.mixed(n_text, 80)]
    streams, avails = [], []
    for p in plains:
        for lv, strat in ((6, zlib.Z_DEFAULT_STRATEGY), (9, zlib.Z_FIXED), (1, zlib.Z_HUFFMAN_ONLY)):
            z = corpus.zlib_raw(p, lv, strat, -15)
            cuts = sorted(set(list(range(max(0, len(z) - 48), len(z) + 1)) + list(range(1, len(z), max(1, len(z) // 23)))))
            for c in cuts:
                streams.append(z[:c]); avails.append(len(p))
            for extra in (1, 2, 7, 9):
                streams.append(z + bytes(extra)); avails.append(len(p))
            for d in (-9, -5, -4, -3, -2, -1, 1, 3):
                streams.append(z); avails.append(max(0, len(p) + d))
    for exact in (False, True):
        got = ctx.decompress_batch_host(streams, avails, 0, exact)
        seen = set()
        for z, a, g in zip(streams, avails, got):
            r = orc.decompress(z, a, 0, exact)
            seen.add(r[0])
            if r[0] == 0:
                assert g == r, ("sweep mismatch", exact, len(z), a, g[0], g[2:], r[2:])
            else:
                assert g[0] == r[0], ("sweep verdict mismatch", exact, len(z), a, g[0], r[0])
        assert seen >= {0, 1, 3}, seen


def check_decompress_large(ctx, sizes=(150000, 262144 + 123), levels=(0, 1, 6, 9)):
    """Chunks larger than the resolve kernel's 32 KiB window ring (several wraps), stored blocks longer
    than its staging span (the literal-run path), runs of equal bytes (offset 1, the periodic path)
    and outputs at every 16-byte phase (the chunks sit back to back in one slab)."""
    plains = []
    for k, n in enumerate(sizes):
        plains += [corpus.text(n, 40 + k), corpus.zeros(n + 1), corpus.pattern(n + 2), corpus.rand(n + 3, k), corpus.mixed(n + 5, k),
                   (b"ab" * 40 + corpus.text(300, k) + b"x" * 700) * (n // 1800)]
    for lv in levels:
        zs = [corpus.zlib_raw(p, lv, zlib.Z_DEFAULT_STRATEGY, -15) for p in plains]
        got = ctx.decompress_batch_host(zs, [len(p) for p in plains], 0)
        for p, g in zip(plains, got):
            assert g[0] == 0 and g[3] == len(p) and g[1] == p, ("large chunk mismatch", lv, len(p), g[0])


def check_packed_round_trip(ctx, n_chunks=300, seed=9, fmts=(0, 2), level=6):
    """The packed host forms: offsets are 16-byte aligned and ascending, the packed streams equal what the
    unpacked call produces, a too small buffer is reported (not overrun), and the packed decompress call
    returns the inputs."""
    rng = random.Random(seed)
    chunks = [corpus.text(rng.choice([0, 1, 100, 3000, 20000, 65536]), i) if i % 3 else corpus.mixed(rng.randrange(1, 30000), i) for i in range(n_chunks)]
    for fmt in fmts:
        packed, offs, sizes = ctx.compress_batch_host_packed(chunks, level, fmt)
        plain = ctx.compress_batch_host(chunks, level, fmt)
        assert len(offs) == n_chunks + 1 and offs[0] == 0 and offs[-1] == len(packed)
        for i, c in enumerate(chunks):
            assert offs[i] % 16 == 0 and offs[i] + sizes[i] <= offs[i + 1] <= offs[i] + sizes[i] + 15
            assert packed[offs[i]:offs[i] + sizes[i]] == plain[i], ("packed stream differs", fmt, i)
        assert ctx.compress_batch_host_packed(chunks, level, fmt, out_avail=len(packed) - 1) is None
        got = ctx.decompress_batch_host_packed(packed, offs, sizes, [len(c) for c in chunks], fmt)
        for g, c in zip(got, chunks):
            assert g[0] == 0 and g[1] == c
    assert ctx.compress_batch_host_packed([], level, 0)[1] == [0]


def check_inputs_with_unmapped_gaps(ctx):
    """Independently allocated input buffers with an unmapped page between them: the host forms must read
    the buffers they were given and nothing else (a whole-span copy would fault)."""
    import ctypes
    import mmap
    page = mmap.PAGESIZE
    m = mmap.mmap(-1, 5 * page)
    base = ctypes.addressof(ctypes.c_char.from_buffer(m))
    libc = ctypes.CDLL(None, use_errno=True)
    libc.mprotect.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int]
    a = corpus.text(page, 1)
    b = corpus.text(page, 2)
    m[0:page] = a
    m[2 * page:3 * page] = b
    assert libc.mprotect(base + page, page, 0) == 0      # PROT_NONE between the two buffers
    assert libc.mprotect(base + 3 * page, 2 * page, 0) == 0
    try:
        n = 2
        ptrs = (ctypes.c_void_p * n)(base, base + 2 * page)
        sizes = (ctypes.c_size_t * n)(page, page)
        bound = ctx.l.libdeflate_gzip_compress_bound(None, page)
        out = ctypes.create_string_buffer(2 * bound)
        optrs = (ctypes.c_void_p * n)(ctypes.addressof(out), ctypes.addressof(out) + bound)
        osz = (ctypes.c_size_t * n)(bound, bound)
        res = (ctypes.c_size_t * n)()
        ctx._check(ctx.l.libdeflate_b200_compress_batch_host(ctx.h, 2, 6, ptrs, sizes, optrs, osz, res, n), "compress_batch_host")
        z = [out.raw[:res[0]], out.raw[bound:bound + res[1]]]
        assert zlib.decompress(z[0], 31) == a and zlib.decompress(z[1], 31) == b
        # and the same layout on the input side of decompress
        m[0:len(z[0])] = z[0]
        m[2 * page:2 * page + len(z[1])] = z[1]
        isz = (ctypes.c_size_t * n)(len(z[0]), len(z[1]))
        dst = ctypes.create_string_buffer(2 * page)
        dptrs = (ctypes.c_void_p * n)(ctypes.addressof(dst), ctypes.addressof(dst) + page)
        dav = (ctypes.c_size_t * n)(page, page)
        rr = (ctypes.c_int32 * n)()
        ao = (ctypes.c_size_t * n)()
        ctx._check(ctx.l.libdeflate_b200_decompress_batch_host(ctx.h, 2, 0, ptrs, isz, dptrs, dav, None, ao, rr, n), "decompress_batch_host")
        assert list(rr) == [0, 0] and dst.raw == a + b
    finally:
        libc.mprotect(base + page, page, 3)
        libc.mprotect(base + 3 * page, 2 * page, 3)


def check_decompress_in_waves(ctx, orc, n_chunks=90):
    """The token scratch between the two inflate kernels is handed out in waves of consecutive chunks; with a 1 MB
    budget this batch needs many of them (and one chunk is larger than the whole budget).  Same results either way."""
    import os
    plains = [corpus.text(20000 + 137 * i, i) if i % 4 else corpus.mixed(9000 + i, i) for i in range(n_chunks)]
    plains[n_chunks // 2] = corpus.text(1500000, 5)
    zs = [corpus.zlib_raw(p, 6, zlib.Z_DEFAULT_STRATEGY, 15) for p in plains]
    zs[3] = zs[3][:len(zs[3]) // 2]                 # a truncated stream in the middle of a wave
    old = os.environ.get("LIBDEFLATE_B200_TOKEN_BUDGET_MB")
    os.environ["LIBDEFLATE_B200_TOKEN_BUDGET_MB"] = "1"
    try:
        got = ctx.decompress_batch_host(zs, [len(p) for p in plains], 1)
    finally:
        if old is None:
            del os.environ["LIBDEFLATE_B200_TOKEN_BUDGET_MB"]
        else:
            os.environ["LIBDEFLATE_B200_TOKEN_BUDGET_MB"] = old
    for i, (p, z, g) in enumerate(zip(plains, zs, got)):
        o = orc.decompress(z, len(p), 1)
        assert g[0] == o[0] and (o[0] != 0 or g == o), ("wave mismatch", i, g[0], o[0])
    assert got[3][0] != 0 and got[4][0] == 0


def gzip_member(plain, flg, level=6, extra=b"EXTRA-field", name=b"file name.txt", comment=b"a comment"):
    """A gzip member with the optional header fields selected by FLG (RFC 1952 2.3: FTEXT 1, FHCRC 2, FEXTRA 4,
    FNAME 8, FCOMMENT 16), built by hand around a zlib-made raw stream."""
    import struct
    hdr = bytes([0x1f, 0x8b, 8, flg, 0, 0, 0, 0, 0, 255])
    if flg & 4:
        hdr += struct.pack("<H", len(extra)) + extra
    if flg & 8:
        hdr += name + b"\0"
    if flg & 16:
        hdr += comment + b"\0"
    if flg & 2:
        hdr += struct.pack("<H", zlib.crc32(hdr) & 0xffff)
    body = corpus.zlib_raw(plain, level, zlib.Z_DEFAULT_STRATEGY, -15)
    return hdr + body + struct.pack("<II", zlib.crc32(plain), len(plain) & 0xffffffff), len(hdr)


def gzip_header_cases():
    """(plain, gzip stream): every combination of the optional header fields, cut inside each of them, reserved
    FLG bits, a missing NUL, empty and long fields."""
    plain = corpus.text(3000, 7)
    cases = []
    for flg in range(32):
        z, hlen = gzip_member(plain, flg)
        cases.append(z)
        cases.append(z + b"trailing garbage")                      # actual_in stops at the member's end
        for cut in sorted(set([10, 11, 12, hlen - 1, hlen, hlen + 1, len(z) - 9, len(z) - 8, len(z) - 1])):
            if 0 < cut < len(z):
                cases.append(z[:cut])
    for bad in (0x20, 0x40, 0x80, 0xE0):
        cases.append(gzip_member(plain, 0)[0][:3] + bytes([bad]) + gzip_member(plain, 0)[0][4:])
    z, _ = gzip_member(plain, 8, name=b"x" * 40)
    cases.append(z[:10] + z[10:].replace(b"\0", b"\1", 1))          # FNAME never terminated before the data runs out?
    cases.append(gzip_member(b"", 4 | 8 | 16 | 2)[0])                # empty payload behind a full header
    z, _ = gzip_member(plain, 4, extra=b"")                          # XLEN = 0
    cases.append(z)
    z, _ = gzip_member(plain, 4, extra=b"q" * 300)
    cases.append(z)
    cases.append(z[:12 + 100])                                      # cut inside FEXTRA
    return [(plain, z) for z in cases]


def check_gzip_optional_fields(ctx, orc, ref_answers=None):
    """ref: lib/gzip_decompress.c:66-98 -- FEXTRA / FNAME / FCOMMENT / FHCRC (and FTEXT) in every combination are
    skipped with bounds checks; reserved FLG bits, truncation inside any field, a missing NUL and a header that leaves
    fewer than 8 bytes for the trailer are BAD_DATA.  Verdicts, actual_in and bytes must equal the oracle's (and,
    given `ref_answers`, the unmodified reference's answers for gzip_header_cases())."""
    import reference_answers as ra
    cases = gzip_header_cases()
    plain = cases[0][0]
    got = ctx.decompress_batch_host([z for _, z in cases], [len(plain)] * len(cases), 2)
    seen = set()
    for k, ((_, z), g) in enumerate(zip(cases, got)):
        o = orc.decompress(z, len(plain), 2)
        assert g[0] == o[0] and (o[0] != 0 or g == o), ("gzip header case", z[:24].hex(), g[0], o[0], g[2:], o[2:])
        if ref_answers is not None:
            r = ref_answers[k]
            assert r[0] == o[0] and (o[0] != 0 or r == ra.outcome(o)), ("oracle vs reference", z[:24].hex(), r[0], o[0])
        seen.add(o[0])
    assert seen >= {0, 1}, seen


def fuzz_cases(n_cases, seed, max_size=20000):
    rng = random.Random(seed)
    base = []
    for n in (0, 1, 10, 300, 3000, max_size):
        for name, v in corpus.all_classes(n, n + 1).items():
            for fmt, wb in ((0, -15), (1, 15), (2, 31)):
                base.append((fmt, v, corpus.zlib_raw(v, rng.choice([1, 6, 9]),
                                                     rng.choice([zlib.Z_DEFAULT_STRATEGY, zlib.Z_FIXED, zlib.Z_HUFFMAN_ONLY]), wb)))
    cases = []
    for _ in range(n_cases):
        fmt, v, z = rng.choice(base)
        z = bytearray(z)
        mode = rng.randrange(6)
        if mode == 0 and len(z):
            for _ in range(rng.randint(1, 3)):
                z[rng.randrange(len(z))] ^= 1 << rng.randrange(8)
        elif mode == 1:
            z = z[:rng.randrange(len(z) + 1)]
        elif mode == 2:
            z += bytes(rng.randrange(256) for _ in range(rng.randint(1, 20)))
        elif mode == 3 and len(z):
            p = rng.randrange(len(z))
            z[p:p + rng.randint(1, 4)] = bytes(rng.randrange(256) for _ in range(rng.randint(0, 4)))
        avail = rng.choice([len(v), len(v), len(v) + rng.randint(0, 100), max(0, len(v) - rng.randint(1, 50)),
                            rng.randint(0, 2 * len(v) + 10)])
        cases.append((fmt, bytes(z), avail, rng.random() < 0.3))
    return cases


def check_decompress_fuzz(ctx, checker, cases):
    """checker.decompress() is the oracle (or the reference); verdicts, byte counts and
    bytes must agree for every mutated stream."""
    n_by_verdict = {}
    for fmt in (0, 1, 2):
        for exact in (False, True):
            sel = [c for c in cases if c[0] == fmt and c[3] == exact]
            if not sel:
                continue
            got = ctx.decompress_batch_host([c[1] for c in sel], [c[2] for c in sel], fmt, exact)
            for c, g in zip(sel, got):
                r = checker.decompress(c[1], c[2], fmt, exact)
                n_by_verdict[r[0]] = n_by_verdict.get(r[0], 0) + 1
                if r[0] == 0:
                    assert g == r, ("fuzz mismatch", fmt, exact, len(c[1]), c[2], g[0], g[2:], r[2:], c[1][:32].hex())
                else:
                    assert g[0] == r[0], ("fuzz verdict mismatch", fmt, exact, len(c[1]), c[2], g[0], r[0], c[1][:32].hex())
    return n_by_verdict


def check_compress_round_trip(ctx, orc, chunks, levels=(1, 6, 9), fmts=(0, 1, 2)):
    """Compressed bytes are not contractual (libdeflate.h:76-83); what is: the stream inflates
    back to the input with the oracle AND zlib, it fits *_compress_bound(), an exactly sized
    output buffer works and one byte less returns 0.  Returns the compressed sizes, format by
    format, level by level, chunk by chunk."""
    wbits = {0: -15, 1: 15, 2: 31}
    sizes = []
    for fmt in fmts:
        for lvl in levels:
            zs = ctx.compress_batch_host(chunks, lvl, fmt)
            for c, z in zip(chunks, zs):
                assert z is not None, ("did not fit its bound", fmt, lvl, len(c))
                assert len(z) <= orc.l.oracle_compress_bound(fmt, len(c)), (fmt, lvl, len(c), len(z))
                r = orc.decompress(z, len(c), fmt)
                assert r[0] == 0 and r[1] == c and r[2] == len(z), ("oracle cannot inflate it", fmt, lvl, len(c))
                assert zlib.decompress(z, wbits[fmt]) == c
                sizes.append(len(z))
            # exact fit and one-byte-short (same streams are deterministic)
            exact = [ctx.compress_batch_host([c], lvl, fmt, out_avail=len(z))[0] for c, z in list(zip(chunks, zs))[:3]]
            assert all(e == z for e, z in zip(exact, zs)), ("exact-size buffer failed", fmt, lvl)
            short = [ctx.compress_batch_host([c], lvl, fmt, out_avail=len(z) - 1)[0] for c, z in list(zip(chunks, zs))[:3]]
            assert all(s is None for s in short), ("short buffer did not return 0", fmt, lvl)
    return sizes


def check_host_pipeline(library, ctx, n=2304, chunk=4096):
    """Large, address-ordered host batches take the pipelined (sub-batched, 3-stream) path of
    libdeflate_b200_*_batch_host; results must equal the plain path's."""
    import ctypes
    import numpy as np
    import bench
    synth = bench.load_synth()
    buf = (ctypes.c_uint8 * (n * chunk))()
    synth.synth_fill(buf, chunk, 0, n, 6, 4)
    raw = bytes(buf)
    inp = np.frombuffer(raw, dtype=np.uint8).copy()
    bound = library.libdeflate_gzip_compress_bound(None, chunk)
    comp = np.zeros(n * bound, dtype=np.uint8)
    idx = np.arange(n, dtype=np.uint64)
    ip = (inp.ctypes.data + idx * chunk).astype(np.uint64)
    isz = np.full(n, chunk, dtype=np.uint64)
    cp = (comp.ctypes.data + idx * bound).astype(np.uint64)
    cav = np.full(n, bound, dtype=np.uint64)
    csz = np.zeros(n, dtype=np.uint64)
    rc = library.libdeflate_b200_compress_batch_host(ctx.h, 2, 6, ip.ctypes.data, isz.ctypes.data, cp.ctypes.data,
                                                     cav.ctypes.data, csz.ctypes.data, n)
    assert rc == 0 and (csz > 0).all()
    for i in (0, 1, n // 2, n - 1):
        assert zlib.decompress(comp[i * bound:i * bound + int(csz[i])].tobytes(), 31) == raw[i * chunk:(i + 1) * chunk]
    out = np.zeros(n * chunk, dtype=np.uint8)
    op = (out.ctypes.data + idx * chunk).astype(np.uint64)
    oav = np.full(n, chunk, dtype=np.uint64)
    aout = np.zeros(n, dtype=np.uint64)
    res = np.zeros(n, dtype=np.int32)
    rc = library.libdeflate_b200_decompress_batch_host(ctx.h, 2, 0, cp.ctypes.data, csz.ctypes.data, op.ctypes.data,
                                                       oav.ctypes.data, None, aout.ctypes.data, res.ctypes.data, n)
    assert rc == 0 and (res == 0).all() and (aout == chunk).all()
    assert out.tobytes() == raw
    # the packed forms take the same sub-batched path: same streams, offsets consistent, round trip exact
    packed = np.zeros(n * (bound + 16), dtype=np.uint8)
    offs = np.zeros(n + 1, dtype=np.uint64)
    psz = np.zeros(n, dtype=np.uint64)
    rc = library.libdeflate_b200_compress_batch_host_packed(ctx.h, 2, 6, ip.ctypes.data, isz.ctypes.data, n, packed.ctypes.data,
                                                            packed.size, offs.ctypes.data, psz.ctypes.data)
    assert rc == 0 and (psz == csz).all() and (offs[:-1] % 16 == 0).all() and (np.diff(offs) >= psz).all() and (np.diff(offs) < psz + 16).all()
    for i in (0, 1, n // 2, n - 1):
        assert packed[int(offs[i]):int(offs[i]) + int(psz[i])].tobytes() == comp[i * bound:i * bound + int(csz[i])].tobytes()
    out2 = np.zeros(n * chunk, dtype=np.uint8)
    op2 = (out2.ctypes.data + idx * chunk).astype(np.uint64)
    res[:] = -1
    rc = library.libdeflate_b200_decompress_batch_host_packed(ctx.h, 2, 0, packed.ctypes.data, offs.ctypes.data, psz.ctypes.data, n,
                                                              op2.ctypes.data, oav.ctypes.data, None, aout.ctypes.data, res.ctypes.data)
    assert rc == 0 and (res == 0).all() and out2.tobytes() == raw


def boundary_chunks():
    """Inputs whose compressible/incompressible seams sit a few bytes off the compressor's 16 KiB pass and
    32 KiB block boundaries: a match that runs across a block end next to a block that is emitted stored
    (regression: the stored block must cover exactly the bytes its tokens would have covered)."""
    import corpus
    out = []
    k = 0
    for seam in (16384, 32768, 49152, 65536, 98304):
        for d in (-9, -1, 0, 1, 8, 100, 257):
            k += 1
            a = seam + d
            out.append(corpus.text(a, k) + corpus.rand(40000 - (k % 3) * 7001, k))
            out.append(corpus.rand(a, k) + corpus.text(33000 + k, k) + corpus.rand(17000, k + 1))
    return out


def check_boundary_round_trip(ctx, levels=(1, 6, 9, 12), fmt=0, every=1):
    chunks = boundary_chunks()[::every]
    wbits = {0: -15, 1: 15, 2: 31}[fmt]
    for lvl in levels:
        zs = ctx.compress_batch_host(chunks, lvl, fmt)
        for c, z in zip(chunks, zs):
            assert z is not None, ("did not fit its bound", lvl, len(c))
            assert zlib.decompress(z, wbits) == c, ("round trip", lvl, len(c))


def check_random_mix_round_trip(ctx, seed=1, rounds=3, per_round=8):
    """Randomised sizes / content mixes / levels / formats: compress, inflate with zlib AND with our own
    decompressor.  (The seam cases above were found with this kind of sweep.)"""
    import random
    import corpus
    rng = random.Random(seed)
    gens = [corpus.text, corpus.rand, lambda n, s: corpus.zeros(n), lambda n, s: corpus.pattern(n), corpus.mixed]
    for _ in range(rounds):
        chunks = []
        for _k in range(per_round):
            total = rng.choice([0, 1, 7, 100, 3000, 16384, 20000, 32768, 40000, 65536, 70000, 100000])
            total = max(0, total + rng.randint(-40, 40)) if total > 50 else total
            parts, left = [], total
            while left > 0:
                n = min(left, rng.choice([5, 50, 500, 4000, 16000, 16384, 33000, 70000]))
                parts.append(rng.choice(gens)(n, rng.randint(0, 10 ** 6))[:n])
                left -= n
            chunks.append(b"".join(parts))
        lvl = rng.choice(range(13))
        fmt = rng.choice([0, 1, 2])
        wbits = {0: -15, 1: 15, 2: 31}[fmt]
        zs = ctx.compress_batch_host(chunks, lvl, fmt)
        for c, z in zip(chunks, zs):
            assert z is not None and zlib.decompress(z, wbits) == c, ("round trip", lvl, fmt, len(c))
        outs = ctx.decompress_batch_host(zs, [len(c) for c in chunks], fmt)
        for c, o in zip(chunks, outs):
            assert o[0] == 0 and o[1] == c, ("own inflate", lvl, fmt, len(c))


def bgzf_reference_file(data, level=6, block=65280):
    """A BGZF file made with Python's zlib only (what bgzip / htslib write): test input for the decompressor."""
    import struct
    out = []
    for off in range(0, len(data), block):
        piece = data[off:off + block]
        co = zlib.compressobj(level, zlib.DEFLATED, -15)
        payload = co.compress(piece) + co.flush()
        bsize = 18 + len(payload) + 8
        out.append(b"\x1f\x8b\x08\x04\0\0\0\0\0\xff\x06\0BC\x02\0" + struct.pack("<H", bsize - 1) + payload
                   + struct.pack("<II", zlib.crc32(piece), len(piece)))
    out.append(bytes([0x1f, 0x8b, 8, 4, 0, 0, 0, 0, 0, 0xff, 6, 0, 66, 67, 2, 0, 27, 0, 3, 0, 0, 0, 0, 0, 0, 0, 0, 0]))
    return b"".join(out)


def check_bgzf(ctx, sizes=(0, 1, 65279, 65280, 65281, 200000), levels=(1, 6)):
    """One buffer <-> blocked gzip file: any gunzip reads ours, we read bgzip-style files, malformed files are
    refused, too-small buffers are reported."""
    import gzip
    import corpus
    for k, n in enumerate(sizes):
        data = corpus.mixed(n, k) if k % 2 else corpus.text(n, k)
        for lvl in levels:
            f = ctx.bgzf_compress(data, lvl)
            assert f is not None and len(f) <= ctx.l.libdeflate_b200_bgzf_compress_bound(n)
            assert gzip.decompress(f) == data                      # an ordinary multi-member gzip file
            assert f.endswith(bgzf_reference_file(b""))             # the BGZF end-of-file member
            assert ctx.bgzf_decompress(f, n) == (0, data)
            if n:
                assert ctx.bgzf_decompress(f, n - 1)[0] == 3       # LIBDEFLATE_INSUFFICIENT_SPACE
                assert ctx.bgzf_compress(data, lvl, out_avail=len(f) - 1) is None
        ref = bgzf_reference_file(data)
        assert ctx.bgzf_decompress(ref, n + 10) == (0, data)
        if n > 100:
            bad = bytearray(ref)
            bad[len(bad) // 2] ^= 0x55                              # payload / CRC damage
            assert ctx.bgzf_decompress(bytes(bad), n)[0] == 1      # LIBDEFLATE_BAD_DATA
            assert ctx.bgzf_decompress(gzip.compress(data), n)[0] == 1   # plain gzip has no BC subfield
            assert ctx.bgzf_decompress(ref[:-40], n)[0] == 1       # truncated
    assert ctx.bgzf_decompress(b"", 10)[0] == 1                    # an empty file is not a gzip file
