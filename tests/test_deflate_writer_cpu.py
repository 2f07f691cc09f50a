"""The deflate stream writer (tests/deflate_writer.py) and its catalogue of edge streams, checked on the CPU: every valid
stream decodes to the bytes the writer meant, in the oracle and in Python's zlib; every invalid one is "Corrupted data
stream" in the oracle.  The GPU tests take the catalogue's expected results from the oracle alone."""
import zlib

import pytest

import deflate_writer as dw
from oracle import zipc_oracle as zo

CASES = dw.all_cases()


def test_bits_and_codes_follow_rfc1951():
    w = dw.Writer()
    w.bits(0b101, 3)          # LSB first: 1, 0, 1
    w.code(0b110, 3)          # MSB first: 1, 1, 0
    w.bits(0b11, 2)
    assert w.finish() == bytes([0b11011101])
    # RFC 1951 3.2.2: lengths (3, 3, 3, 3, 3, 2, 4, 4) for A .. H
    assert dw.canonical([3, 3, 3, 3, 3, 2, 4, 4]) == {0: (0b010, 3), 1: (0b011, 3), 2: (0b100, 3), 3: (0b101, 3),
                                                       4: (0b110, 3), 5: (0b00, 2), 6: (0b1110, 4), 7: (0b1111, 4)}
    fixed = dw.canonical(dw.FIXED_LIT)
    assert fixed[0] == (0b00110000, 8) and fixed[144] == (0b110010000, 9) and fixed[256] == (0, 7) and fixed[280] == (0b11000000, 8)


def test_writer_output_matches_zlib_for_fixed_and_stored_blocks():
    """a fixed block and a stored block: the bytes zlib writes for the same content"""
    w = dw.Writer()
    w.fixed(True)
    w.literals(b"a")
    w.eob()
    c = zlib.compressobj(9, zlib.DEFLATED, -15, 9, zlib.Z_FIXED)
    assert w.finish() == c.compress(b"a") + c.flush()
    w = dw.Writer()
    w.stored(b"hello", True)
    c = zlib.compressobj(0, zlib.DEFLATED, -15)
    assert w.finish() == c.compress(b"hello") + c.flush()


def test_rle_symbols_spell_the_lengths():
    for lengths in ([0] * 300, [5] * 40 + [0] * 7 + [3] * 2 + [0] * 150, [8] * 286 + [5] * 30, [1, 0, 0, 1, 1, 1, 1]):
        spelled = []
        for s, e in dw.rle_symbols(lengths):
            if s < 16:
                spelled.append(s)
            elif s == 16:
                spelled += [spelled[-1]] * (3 + e)
            else:
                spelled += [0] * ((3 if s == 17 else 11) + e)
        assert spelled == lengths


@pytest.mark.parametrize("case", CASES, ids=[c.name for c in CASES])
def test_catalogue_stream_in_the_oracle_and_zlib(case):
    if case.valid:
        out, _ = zo.inflate_and_crc(case.stream, None)
        assert out == case.out
        assert zo.inflate(case.stream, len(case.out)) == case.out
        if case.name.startswith(("clen_single", "lit_only_end_of_block", "dist_single_code_bit_0", "hclen_5")):
            return   # (zlib refuses some incomplete codes the reference accepts)
        d = zlib.decompressobj(-15)
        assert d.decompress(case.stream) == case.out and d.eof
    else:
        with pytest.raises(zo.OracleError) as e:
            zo.inflate(case.stream)
        assert e.value.status == zo.ERR_CORRUPTED


def test_catalogue_covers_both_sides_of_each_rule():
    names = {c.name: c.valid for c in CASES}
    for ok, bad in (("hlit_286", "hlit_287"), ("hdist_30", "hdist_31"), ("rle_18_fills_exactly", "rle_18_overruns_by_one"),
                    ("rle_16_fills_exactly", "rle_16_overruns_by_one"), ("lit_only_end_of_block", "lit_only_end_of_block_bit_1"),
                    ("dist_single_code_bit_0", "dist_single_code_bit_1"), ("dist_first_match_equal", "dist_first_match_plus_1"),
                    ("dist_after_stored_equal", "dist_after_stored_plus_1"), ("dist_second_block_equal", "dist_second_block_plus_1")):
        assert names[ok] and not names[bad]
    adler = [c for c in CASES if c.name.startswith("adler_") and c.name.rsplit("_", 1)[1].isdigit()]
    assert sorted({len(c.out) for c in adler}) == list(dw.ADLER_LENGTHS) and all(set(c.out) <= {0xFF} for c in adler)
