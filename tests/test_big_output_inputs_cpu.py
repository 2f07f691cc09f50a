"""The builders of big_output_inputs.py, no GPU: each one at a few MiB of output (the same construction with fewer copies of
its unit) against zlib, the oracle and par_inflate_model, and each full-size stream's properties read off its structure
without decoding it."""
import zlib

import numpy as np
import pytest

import big_output_inputs as bo
import par_inflate_model as pm
from oracle import zipc_oracle as zo

NAMES = list(bo.BUILDERS)
TWO32 = 1 << 32


def _full(name):
    return [(name, t) for t in (bo.LEN_JUST_OVER, bo.LEN_LONG) if not (name == "big_block" and t == bo.LEN_JUST_OVER)]


FULL = [x for n in NAMES for x in _full(n)]


@pytest.fixture(scope="module", params=NAMES)
def small(request):
    b = bo.BUILDERS[request.param](bo.small_total(request.param))
    return b, b.stream()


def test_small_stream_outputs_the_tiled_prefix(small):
    b, raw = small
    want = bo.expected(b.total)
    assert np.array_equal(np.frombuffer(zlib.decompress(raw, -15), dtype=np.uint8), want)
    out = zo.inflate(raw)
    assert np.array_equal(np.frombuffer(out, dtype=np.uint8), want)
    assert zlib.crc32(out) == bo.expected_crc32(b.total)


def test_small_stream_adler_model(small):
    """the block fold in both modes: RFC 1950 is zlib.adler32 of the output; the reference's word is what the oracle's
    zlib_decompress finds (it raises on any other trailer)"""
    b, raw = small
    out = zlib.decompress(raw, -15)
    assert bo.adler32_blocks(b, "rfc") == zlib.adler32(out)
    ref = bo.adler32_blocks(b, "ref")
    back, found = zo.zlib_decompress(bo.zlib_wrap(raw, ref))
    assert back == out and found == ref


def test_small_stream_blocks_and_finder(small):
    """the block table is the model's walk, the finder hits exactly the non-final dynamic blocks (no false start anywhere in
    the head, the unit or the tail), and the model's plan is the one chunk_plan predicts"""
    b, raw = small
    w = pm.walk(raw)
    assert w.error is None
    bits, outs, btype = b.block_table()
    assert [x.start for x in w.blocks] == bits.tolist()
    assert [x.btype for x in w.blocks] == btype.tolist()
    assert [x.out_len for x in w.blocks] == b.block_lengths().tolist()
    hits = pm.valid_starts(raw)
    assert hits.tolist() == bits[:-1][btype[:-1] == 2].tolist()
    pl = pm.plan(raw, w=w, hits=hits)
    if b.name == "expand":
        assert pl.outcome == "no_start"
    else:
        assert pl.outcome == "parallel" and pl.recuts == 0
        starts, out_len, _, _ = bo.chunk_plan(b)
        assert [c.start for c in pl.chunks] == starts.tolist()
        assert [c.out_len for c in pl.chunks] == out_len.tolist()


@pytest.mark.parametrize("name,total", FULL)
def test_full_stream_properties(name, total):
    b = bo.BUILDERS[name](total)
    _, outs, btype = b.block_table()
    lens = b.block_lengths()
    assert b.total == total == int(lens.sum()) and total > TWO32
    # the tiled unit starts and ends on a byte boundary and holds whole blocks or whole 32 KiB periods
    assert b.unit_bits % 8 == 0 and len(b.mid) == b.unit_bits // 8 and b.copies > 1000
    assert b.head_bits >= 8 * (bo.PERIOD + 5)
    # matches copy bytes in [2^32, 2^32 + 32768): there a 32-bit output position would see a distance of 32768 reach
    # before the start of the output
    if total > TWO32 + bo.PERIOD:
        assert b.match_bytes(TWO32, TWO32 + bo.PERIOD) >= bo.PERIOD // 2
    if name == "expand":
        assert b.match_bytes(TWO32, min(total, TWO32 + bo.PERIOD)) == min(total - TWO32, bo.PERIOD)
    assert b.match_bytes(0, bo.PERIOD) == 0
    if name == "expand":
        # one fixed block after the prefix, ~80-fold: over the 24-fold budget of a speculative chunk, and nothing to find
        assert btype.tolist() == [0, 1] and lens[1] == total - bo.PERIOD
        assert b.unit_out / len(b.mid) > 24 + 65536 / 8192
        return
    starts, out_len, nbytes, spec_cap = bo.chunk_plan(b)
    budget = 24 * nbytes + 65536
    assert (out_len <= budget).all()                 # every chunk under its symbol budget
    assert spec_cap <= 6 << 30                       # the whole stream under the symbols the decoder sets aside
    if name == "spread":
        assert (lens[1:] <= bo.SMALL_OUT).all() and len(starts) > 16000
        assert (out_len[1:] > 16 * nbytes[1:]).all()  # (and expanding enough that 4 GiB fit those symbols)
    else:
        assert int(lens.max()) >= TWO32 and btype[int(np.argmax(lens))] == 2
        assert len(starts) == 3 and out_len[1] >= TWO32 and out_len[1] <= 24 * nbytes[1]


def test_zip64_archive_read_by_cpython(small):
    """the hand-built ZIP64 archive: CPython's zipfile reads its directory at full size and the member at small size"""
    import io
    import zipfile
    b, raw = small
    arc, at = bo.zip64_archive(raw, b.total, bo.expected_crc32(b.total))
    with zipfile.ZipFile(io.BytesIO(arc)) as z:
        (info,) = z.infolist()
        assert (info.filename, info.compress_type, info.file_size, info.compress_size) == ("big.bin", 8, b.total, len(raw))
        assert np.array_equal(np.frombuffer(z.read("big.bin"), dtype=np.uint8), bo.expected(b.total))
    assert arc[at:at + len(raw)] == raw
    big = bo.spread(bo.LEN_LONG)
    full = big.stream()
    arc, at = bo.zip64_archive(full, big.total, 0)
    with zipfile.ZipFile(io.BytesIO(arc)) as z:
        (info,) = z.infolist()
        assert (info.file_size, info.compress_size, info.header_offset) == (big.total, len(full), 0)
