"""Golden fixtures (tests/golden/, generated from the UNMODIFIED reference by
make_fixtures.py) against the oracle and, through the emulator, the kernel logic."""
import json
import os
import random

import deflate_asm as da
import reference_answers as ra

HERE = os.path.dirname(os.path.abspath(__file__))


def _known():
    return json.load(open(os.path.join(HERE, "golden", "known_answer.json")))


def test_oracle_known_answers(oracle):
    for k in _known():
        r = oracle.decompress(bytes.fromhex(k["stream"]), k["out_avail"], 0)
        assert r[0] == k["result"], k["name"]
        if k["result"] == 0:
            assert r[1] == bytes.fromhex(k["output"]), k["name"]


def test_oracle_inflates_reference_compressor_output(oracle):
    for fmt, plain, z in ra.fixture_streams():
        r = oracle.decompress(z, len(plain), fmt)
        assert r[0] == 0 and r[1] == plain and r[2] == len(z)


def test_kernel_logic_known_answers_emulated(emu_ctx):
    ka = _known()
    got = emu_ctx.decompress_batch_host([bytes.fromhex(k["stream"]) for k in ka], [k["out_avail"] for k in ka], 0)
    for k, g in zip(ka, got):
        assert g[0] == k["result"], k["name"]
        if k["result"] == 0:
            assert g[1] == bytes.fromhex(k["output"]), k["name"]


def test_kernel_logic_reference_streams_emulated(emu_ctx):
    streams = ra.fixture_streams()
    for fmt in (0, 1, 2):
        sel = [s for s in streams if s[0] == fmt]
        got = emu_ctx.decompress_batch_host([s[2] for s in sel], [len(s[1]) for s in sel], fmt)
        for g, s in zip(got, sel):
            assert g[0] == 0 and g[1] == s[1] and g[2] == len(s[2])


def test_kernel_logic_odd_codes_emulated(emu_ctx, oracle):
    """Arbitrary complete codes with 15-bit codewords: exercises subtables and the
    shared-memory-overflow path of the table builder."""
    rng = random.Random(2)
    streams = [da.odd_code_stream(rng, n_tokens=rng.randint(1, 800)) for _ in range(120)]
    got = emu_ctx.decompress_batch_host([s[0] for s in streams], [len(s[1]) for s in streams], 0)
    for (z, p), g in zip(streams, got):
        o = oracle.decompress(z, len(p), 0)
        assert o[0] == 0 and o[1] == p and g == o
