"""Pins the oracle (oracle/*.c, our restatement) to the UNMODIFIED reference -- through its
answers recorded in tests/golden/reference_answers.npz -- and to zlib, before anything else
trusts it (prompt section 3)."""
import zlib

import corpus
import reference_answers as ra


def test_oracle_checksums_match_reference_and_zlib(oracle):
    cases = ra.checksum_cases()
    for (d, init, a), (ref_crc, ref_adler) in zip(cases, ra.answers("checksums", cases)):
        assert oracle.crc32(d, init) == ref_crc == zlib.crc32(d, init)
        assert oracle.adler32(d, a) == ref_adler == zlib.adler32(d, a)


def test_oracle_decompress_matches_reference_on_valid_streams(oracle):
    cases = ra.valid_stream_cases()
    for (fmt, plain, z), r in zip(cases, ra.answers("valid_streams", cases)):
        o = oracle.decompress(z, len(plain), fmt)
        assert r[0] == 0 and r == ra.outcome(o)


def test_oracle_verdicts_match_reference_on_mutated_streams(oracle):
    seen = {}
    cases = ra.fuzz_cases()
    for (fmt, z, avail, exact), r in zip(cases, ra.answers("fuzz", cases)):
        o = oracle.decompress(z, avail, fmt, exact)
        seen[r[0]] = seen.get(r[0], 0) + 1
        if r[0] == 0:
            assert ra.outcome(o) == r
        else:
            assert o[0] == r[0], (fmt, avail, exact, z[:40].hex())
    assert set(seen) == {0, 1, 2, 3}, seen


def test_oracle_bound_and_stored_blocks_match_reference(oracle):
    cases = [(n, fmt) for n in ra.STORED_SIZES for fmt in (0, 1, 2)]
    for (n, fmt), (ref_bound, ref_stored) in zip(cases, ra.answers("bound_and_stored", cases)):
        assert oracle.l.oracle_compress_bound(fmt, n) == ref_bound
        assert ra.digest(oracle.compress_stored(corpus.rand(n, n), fmt, 0)) == ref_stored
