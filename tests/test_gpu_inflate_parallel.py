"""GPU parity: intra-stream parallel inflate of LARGE foreign streams (no index).  The bar is the same as for every inflate:
output, checksum and status are those of the oracle (and zlib) -- whether the stream was decoded by many warps (block
starts found by scanning, speculative chunks, resolve) or handed back to the one-warp decoder because something did not
check out.  The tests also assert that the parallel path is really taken where it should be."""
import os
import random
import zlib

import numpy as np
import pytest

from oracle import zipc_oracle as zo
from test_gpu_inflate_spec_plan import decode_pinned
from zipc_b200 import _lib, synth
from zipc_b200 import zipc_deflate as zd

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = zd.Context(0)
    zd.set_default_context(c)
    yield c
    zd.set_default_context(None)
    c.close()


def _raw(data: bytes, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, memlevel=8) -> bytes:
    c = zlib.compressobj(level, zlib.DEFLATED, -15, memlevel, strategy)
    return c.compress(data) + c.flush()


def _check(ctx, stream: bytes, data: bytes, expect_parallel=None):
    before = ctx.parallel_streams
    (st, out, crc), = ctx.inflate_batch([stream], [len(data)], _lib.CK_CRC32)
    assert st == 0 and crc == zlib.crc32(data) and out.tobytes() == data
    after = ctx.parallel_streams
    if expect_parallel is True:
        assert after[0] == before[0] + 1, "the stream was not decoded in parallel"
    elif expect_parallel is False:
        assert after[0] == before[0]
    # unknown size: same answer through the sizing pass
    (st, out, crc), = ctx.inflate_batch([stream], [None], _lib.CK_CRC32)
    assert st == 0 and crc == zlib.crc32(data) and out.tobytes() == data


@pytest.mark.parametrize("level", [1, 6, 9])
def test_large_zlib_streams(ctx, level):
    data = synth.text_v1(40 + level, (6 << 20) + 12345).tobytes()
    stream = _raw(data, level)
    assert len(stream) > (1 << 20)
    _check(ctx, stream, data, expect_parallel=True)
    out, crc = zo.inflate_and_crc_32(stream, len(data))  # the oracle agrees (and so does zlib, by construction)
    assert out == data and crc == zlib.crc32(data)


def test_mixed_content_and_block_kinds(ctx):
    """text, incompressible stretches (stored blocks), runs (long matches, distance 1), binary structure; also streams made
    with Z_FIXED (no dynamic block anywhere: nothing to find, serial path) and Z_HUFFMAN_ONLY / Z_RLE.  Each takes the path
    and the passes and chunks of tests/par_inflate_model.py's plan: under Z_RLE and Z_FILTERED the 500,000 zero bytes come
    out of a chunk at more than 24 times its compressed size, and the one-warp decoder takes the stream."""
    rnd = random.Random(9)
    t = synth.text_v1(77, 3 << 20).tobytes()
    parts = [t[:900000], rnd.randbytes(300000), bytes(500000), t[900000:2000000], bytes(range(256)) * 2000, rnd.randbytes(70000), t[2000000:]]
    data = b"".join(parts)
    for level, strategy in ((6, zlib.Z_DEFAULT_STRATEGY), (1, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_RLE), (6, zlib.Z_HUFFMAN_ONLY), (6, zlib.Z_FILTERED)):
        stream = _raw(data, level, strategy)
        plan = decode_pinned(ctx, stream, [len(data), None], chunk=8192, par_min=None)
        assert plan.outcome == ("symbol_budget" if strategy in (zlib.Z_RLE, zlib.Z_FILTERED) else "parallel"), plan.describe()
    plan = decode_pinned(ctx, _raw(t, 6, zlib.Z_FIXED), [len(t), None], chunk=8192, par_min=None)
    assert plan.outcome == "no_start"


def test_stream_made_by_the_oracle_and_by_us(ctx):
    data = synth.text_v1(5, 2_500_000).tobytes()
    _check(ctx, zo.deflate(data, "default"), data, expect_parallel=True)
    cs = zd.deflate(data, level="default").get_ok()
    _check(ctx, cs, data)


def test_small_chunks_and_thresholds(ctx, monkeypatch):
    """the same machinery with tiny chunks and a low threshold: many more boundaries, chunks shorter than a window"""
    monkeypatch.setenv("ZIPC_B200_PAR_MIN", "20000")
    monkeypatch.setenv("ZIPC_B200_PAR_CHUNK", "4096")
    for seed, n in ((1, 300_000), (2, 1_000_000), (3, 70_001)):
        data = synth.text_v1(100 + seed, n).tobytes()
        for level in (1, 6):
            c = zlib.compressobj(level, zlib.DEFLATED, -15, 1)  # memLevel 1: small blocks
            stream = c.compress(data) + c.flush()
            plan = decode_pinned(ctx, stream, [len(data), None], chunk=4096, par_min=20000)
            assert plan.outcome == "parallel" and len(plan.chunks) > 4, plan.describe()
    # the reference's own fixture size at level 9: zlib writes it in two dynamic blocks, and the second is found
    data = synth.text_v1(9, 174_585).tobytes()
    plan = decode_pinned(ctx, _raw(data, 9), [len(data), None], chunk=4096, par_min=20000)
    assert plan.outcome == "parallel" and len(plan.chunks) == 2, plan.describe()


def test_corrupt_large_streams_have_the_reference_status(ctx):
    data = synth.text_v1(6, 3 << 20).tobytes()
    stream = bytearray(_raw(data, 6))
    rnd = random.Random(4)
    cases = []
    for _ in range(12):
        s = bytearray(stream)
        at = rnd.randrange(len(s))
        s[at] ^= 1 << rnd.randrange(8)
        cases.append(bytes(s))
    cases.append(bytes(stream[: len(stream) // 2]))          # truncated
    cases.append(bytes(stream[:1000]) + bytes(stream[5000:]))  # a hole
    cases.append(bytes(stream) + b"trailing bytes are ignored")
    for s in cases:
        for cap in (len(data), len(data) - 1, None):
            try:
                ref = (0, zo.inflate_and_crc_32(s, cap))
            except zo.OracleError as e:
                ref = (e.status, None)
            (st, out, crc), = ctx.inflate_batch([s], [cap], _lib.CK_CRC32)
            assert st == ref[0], (st, ref[0], cap)
            if st == 0:
                assert out.tobytes() == ref[1][0] and crc == ref[1][1]


def test_throughput_sanity_and_batch_mix(ctx):
    """a batch that mixes small members with two large streams: everything comes back in order, large ones in parallel"""
    big1 = synth.text_v1(61, 4 << 20).tobytes()
    big2 = synth.text_v1(62, 3 << 20).tobytes()
    small = [synth.text_v1(200 + i, 5000 + 777 * i).tobytes() for i in range(20)]
    datas = small[:10] + [big1] + small[10:] + [big2]
    streams = [_raw(d, 6) for d in datas]
    before = ctx.parallel_streams
    res = ctx.inflate_batch(streams, [len(d) for d in datas], _lib.CK_CRC32)
    for d, (st, out, crc) in zip(datas, res):
        assert st == 0 and out.tobytes() == d and crc == zlib.crc32(d)
    assert ctx.parallel_streams[0] == before[0] + 2


def test_many_mid_sized_streams_stay_on_the_one_warp_decoder(ctx):
    """The many-warp decoder takes a handful of streams at a time (one lane each): it is chosen where that shortens the call (a
    few mid-sized or large streams, alone or among small ones), not for hundreds of equally large streams, which the one-warp
    decoder takes side by side (148 streams of 1 MiB: 30 ms there, 816 ms one after the other)."""
    data = synth.text_v1(321, 1 << 20).tobytes()
    stream = _raw(data, 6)
    assert len(stream) > 300_000
    before = ctx.parallel_streams
    (st, out, crc), = ctx.inflate_batch([stream], [len(data)], _lib.CK_CRC32)          # alone: in parallel
    assert st == 0 and crc == zlib.crc32(data) and ctx.parallel_streams[0] == before[0] + 1
    mid = synth.text_v1(322, 200_000).tobytes()                                          # 70 KB compressed: alone, in parallel too
    (st, out, crc), = ctx.inflate_batch([_raw(mid, 6)], [len(mid)], _lib.CK_CRC32)
    assert st == 0 and out.tobytes() == mid and ctx.parallel_streams[0] == before[0] + 2
    before = ctx.parallel_streams
    res = ctx.inflate_batch([stream] * 12, [len(data)] * 12, _lib.CK_CRC32)             # a dozen: several at a time, on the lanes
    assert all(st == 0 and crc == zlib.crc32(data) for st, _, crc in res) and res[11][1].tobytes() == data
    assert ctx.parallel_streams[0] == before[0] + 12
    before = ctx.parallel_streams
    res = ctx.inflate_batch([stream] * 240, [len(data)] * 240, _lib.CK_CRC32)           # hundreds of them: side by side, a warp each
    assert all(st == 0 and crc == zlib.crc32(data) for st, _, crc in res) and res[239][1].tobytes() == data
    assert ctx.parallel_streams == before


def test_large_zlib_streams_with_adler32_take_the_many_warp_path(ctx):
    """zlib_decompress / inflate_and_adler_32 of a large stream: decoded by many warps, the Adler-32 folded block by block over
    the block lengths the chunks report -- bit-exact with the reference's per-block fold (signed remainder, state re-packed
    between blocks: zipc_deflate.ml:175-198, 682-690) on data where that differs from RFC 1950."""
    t = np.frombuffer(synth.text_v1(91, 5 << 20).tobytes(), dtype=np.uint8)
    quirk = (t | 0x80).tobytes()[:-333] + b"\xff" * 300_000 + synth.rand_v1(92, 200_001).tobytes() + bytes(70_000)
    text = t.tobytes()
    for data in (text, quirk):
        raw = _raw(data, 6)
        want_out, want_ad = zo.inflate_and_adler_32(raw, len(data))       # the reference's fold over zlib's blocks
        before = ctx.parallel_streams
        (st, out, ad), = ctx.inflate_batch([raw], [len(data)], _lib.CK_ADLER32, _lib.ADLER_REF_COMPAT)
        assert st == 0 and out.tobytes() == data == want_out and ad == want_ad
        assert ctx.parallel_streams[0] == before[0] + 1
        (st, out, ad), = ctx.inflate_batch([raw], [None], _lib.CK_ADLER32, _lib.ADLER_RFC1950)   # sizing pass first
        assert st == 0 and out.tobytes() == data and ad == zlib.adler32(data)
    assert zo.inflate_and_adler_32(_raw(quirk, 6), len(quirk))[1] != zlib.adler32(quirk)         # (the quirk is exercised)
    # the zlib framing on top: a standard stream of quirk data is a checksum mismatch in the reference's flavour, with its pair
    z = zlib.compress(quirk, 6)
    r = zd.zlib_decompress(z)
    try:
        zo.zlib_decompress(z)
        raise AssertionError("the oracle accepted the stream")
    except zo.OracleError as e:
        assert r.is_error() and r.info == (e.extra["expect"], e.extra["found"])
    assert zd.zlib_decompress(z, adler_mode=_lib.ADLER_RFC1950).get_ok() == (quirk, zlib.adler32(quirk))
    # and our own zlib_compress of a large payload (split over CTAs) comes back through it
    ad, zs = zd.zlib_compress(quirk, level="default").get_ok()
    assert zd.zlib_decompress(bytes(zs)).get_ok() == (quirk, ad)
