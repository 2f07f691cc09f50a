"""Host <-> device transfers of the host-pointer entry points, checked against zlib and the oracle.

Pageable host memory travels through a pinned staging ring of 16 MiB chunks; pinned memory, and any copy of 64 KiB or
less, is one DMA.  The sizes here sit on both sides of those two limits.  Ranges of a batch that lie more than a page
apart are uploaded one by one, the pageable ones packed chunk by chunk with zero padding to 16 bytes; the ranges here
cross chunk boundaries and end right before one.  Every host-pointer call that fills an output arena is run twice: into
a pageable arena of more than 32 MiB, and without an arena followed by zipc_b200_fetch.  Both runs must report and
deliver the same."""
import contextlib
import ctypes as C
import io
import zipfile
import zlib

import numpy as np
import pytest

from oracle import zipc_oracle as zo
from zipc_b200 import _lib, synth
from zipc_b200 import zipc_deflate as zd

pytestmark = pytest.mark.gpu

KiB, MiB = 1 << 10, 1 << 20
STAGE = 16 * MiB
SIZES = [64 * KiB - 1, 64 * KiB, 64 * KiB + 1, STAGE - 1, STAGE + 1, 2 * STAGE + 17]
OFFSETS = [0, 1, 15]


@pytest.fixture(scope="module")
def ctx():
    c = zd.Context(0)
    yield c
    c.close()


@contextlib.contextmanager
def pinned(ctx, size):
    """a uint8 array over zipc_b200_host_alloc memory"""
    p = C.c_void_p()
    ctx._check(ctx.L.zipc_b200_host_alloc(max(size, 1), C.byref(p)), "host_alloc")
    try:
        yield np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(max(size, 1),))[:size]
    finally:
        ctx.L.zipc_b200_host_free(p)


def P(a, ty):
    return a.ctypes.data_as(C.POINTER(ty))


@pytest.fixture(scope="module")
def blob():
    """random bytes (no two 16 MiB chunks alike) for the checksum and copy tests"""
    return synth.rand_v1(77, 2 * STAGE + 17 + 64)


# ---- whole buffers: checksums and plain copies ---------------------------------------------------------------------------
@pytest.mark.parametrize("size", SIZES)
def test_checksums_of_pageable_and_pinned_buffers(ctx, blob, size):
    L = ctx.L
    with pinned(ctx, size + 16) as pin:
        for off in OFFSETS:
            data = blob[off:off + size]
            want = {"crc": zlib.crc32(data), "rfc": zlib.adler32(data), "ref": zo.adler32(data.tobytes())}
            pageable = np.empty(size + 16, dtype=np.uint8)
            pageable[off:off + size] = data
            pin[off:off + size] = data
            for kind, buf in (("pageable", pageable), ("pinned", pin)):
                p = buf.ctypes.data + off
                crc, rfc, ref = C.c_uint32(), C.c_uint32(), C.c_uint32()
                ctx._check(L.zipc_b200_crc32(ctx.h, p, size, C.byref(crc)), "crc32")
                ctx._check(L.zipc_b200_adler32(ctx.h, p, size, _lib.ADLER_RFC1950, C.byref(rfc)), "adler32")
                ctx._check(L.zipc_b200_adler32(ctx.h, p, size, _lib.ADLER_REF_COMPAT, C.byref(ref)), "adler32")
                got = {"crc": crc.value, "rfc": rfc.value, "ref": ref.value}
                assert got == want, (kind, size, off)


@pytest.mark.parametrize("size", SIZES)
def test_memcpy_round_trips(ctx, blob, size):
    L = ctx.L
    d = C.c_void_p()
    ctx._check(L.zipc_b200_dev_alloc(ctx.h, size, C.byref(d)), "dev_alloc")
    try:
        with pinned(ctx, size) as pin_in, pinned(ctx, size) as pin_out:
            pin_in[:] = blob[5:5 + size]
            for src_kind, src in (("pageable", blob[3:3 + size].copy()), ("pinned", pin_in)):
                ctx._check(L.zipc_b200_memcpy_h2d(ctx.h, d, src.ctypes.data, size), "memcpy_h2d")
                for dst_kind in ("pageable", "pinned"):
                    dst = np.full(size, 0xA5, dtype=np.uint8) if dst_kind == "pageable" else pin_out
                    dst[:] = 0xA5
                    ctx._check(L.zipc_b200_memcpy_d2h(ctx.h, dst.ctypes.data, d, size), "memcpy_d2h")
                    assert np.array_equal(dst, src), (src_kind, dst_kind, size)
    finally:
        L.zipc_b200_dev_free(ctx.h, d)


# ---- ranges copied one by one -------------------------------------------------------------------------------------------
def ragged_ranges():
    """(offset, length) of ranges with gaps of a page or more between them, and the size of the buffer that holds them.  Packed
    with 16-byte padding, as the pageable ones are staged, range 2 crosses the first 16 MiB boundary, range 4 ends 5 bytes
    before the second (its padding fills them) and range 6 crosses the third; zero-length ranges sit in between."""
    lens = [5 * MiB + 3, 0, 12 * MiB + 7, 0, 15 * MiB - 37, 0, 17 * MiB + 1, 1, 15, 0, 17, 4096, 64 * KiB + 3]
    packed = np.cumsum([0] + [(n + 15) & ~15 for n in lens])
    assert packed[2] < STAGE < packed[3] and packed[4] + lens[4] == 2 * STAGE - 5 and packed[6] < 3 * STAGE < packed[7]
    assert sum(lens) > 40 * MiB
    ranges, pos = [], 64
    for i, n in enumerate(lens):
        ranges.append((pos, n))
        pos += n + 4096 + 16 * (i % 3) + i % 5
    return ranges, pos


def test_crc32_batch_of_separate_ranges(ctx):
    ranges, size = ragged_ranges()
    pageable = synth.rand_v1(91, size)
    want = [zlib.crc32(pageable[o:o + n]) for o, n in ranges]
    n = len(ranges)
    lens = np.array([ln for _, ln in ranges], dtype=np.uint64)
    with pinned(ctx, size) as pin:
        pin[:] = pageable
        for mixed in (False, True):  # every range pageable; every other range pinned
            bufs = [pin if mixed and i % 2 else pageable for i in range(n)]
            # a zero-length range may come without a pointer
            ptrs = (C.c_void_p * n)(*[None if ln == 0 and i % 4 == 1 else b.ctypes.data + o for i, ((o, ln), b) in enumerate(zip(ranges, bufs))])
            out = np.zeros(n, dtype=np.uint32)
            ctx._check(ctx.L.zipc_b200_crc32_batch(ctx.h, n, ptrs, P(lens, C.c_size_t), P(out, C.c_uint32)), "crc32_batch")
            assert out.tolist() == want, mixed


# ---- output arenas: staged download vs fetch ----------------------------------------------------------------------------
ARENA_MIN = 32 * MiB


@pytest.fixture(scope="module")
def members():
    """48 members of about 1 MiB, three random for every text one: the compressed outputs pass 32 MiB as well"""
    return [(synth.text_v1 if i % 4 == 0 else synth.rand_v1)(300 + i, MiB + 37 * i) for i in range(48)]


def arena_twice(ctx, call, n, what):
    """call(dst, cap, need, off, len) -> rc, once without an arena (then fetch) and once into a pageable arena of exactly the
    size asked for.  Sizes, offsets, lengths and output bytes must agree; returns the output bytes."""
    runs = []
    for with_arena in (False, True):
        need = C.c_size_t()
        off = np.zeros(max(n, 1), dtype=np.uint64)
        ln = np.zeros(max(n, 1), dtype=np.uint64)
        if with_arena:
            arena = np.full(runs[0]["need"], 0x5A, dtype=np.uint8)
            rc = call(arena.ctypes.data, arena.size, C.byref(need), P(off, C.c_size_t), P(ln, C.c_size_t))
            assert rc == _lib.OK, (what, rc)
        else:
            rc = call(None, 0, C.byref(need), P(off, C.c_size_t), P(ln, C.c_size_t))
            assert rc == _lib.ERR_DST_TOO_SMALL, (what, rc)
            arena = np.full(need.value, 0xC3, dtype=np.uint8)
            ctx._check(ctx.L.zipc_b200_fetch(ctx.h, arena.ctypes.data, arena.size), "fetch")
        assert need.value > ARENA_MIN, what
        outs = [arena[int(off[i]):int(off[i]) + int(ln[i])].tobytes() for i in range(n)]
        runs.append({"need": need.value, "off": off[:n].tolist(), "len": ln[:n].tolist(), "outs": outs})
    a, b = runs
    assert a["need"] == b["need"] and a["off"] == b["off"] and a["len"] == b["len"], what
    assert a["outs"] == b["outs"], what
    return a["outs"]


def test_deflate_batch(ctx, members):
    n = len(members)
    ptrs, lens = zd.Context._ptr_arrays(members)
    seen = []

    def call(dst, cap, need, off, ln):
        ck = np.zeros(n, dtype=np.uint32)
        st = np.full(n, -1, dtype=np.int32)
        rc = ctx.L.zipc_b200_deflate_batch(ctx.h, _lib.LEVEL_DEFAULT, _lib.CK_CRC32, 0, n, ptrs, lens, dst, cap, need, off, ln,
                                           P(ck, C.c_uint32), P(st, C.c_int))
        seen.append((ck.tolist(), st.tolist()))
        return rc
    outs = arena_twice(ctx, call, n, "deflate_batch")
    assert seen[0] == seen[1]
    for m, out, ck, st in zip(members, outs, *seen[0]):
        assert st == 0 and ck == zlib.crc32(m) and zlib.decompress(out, -15) == m.tobytes()


def test_zlib_compress_batch(ctx, members):
    n = len(members)
    ptrs, lens = zd.Context._ptr_arrays(members)
    seen = []

    def call(dst, cap, need, off, ln):
        ad = np.zeros(n, dtype=np.uint32)
        st = np.full(n, -1, dtype=np.int32)
        rc = ctx.L.zipc_b200_zlib_compress_batch(ctx.h, _lib.LEVEL_FAST, _lib.ADLER_RFC1950, n, ptrs, lens, dst, cap, need, off, ln,
                                                 P(ad, C.c_uint32), P(st, C.c_int))
        seen.append((ad.tolist(), st.tolist()))
        return rc
    outs = arena_twice(ctx, call, n, "zlib_compress_batch")
    assert seen[0] == seen[1]
    for m, out, ad, st in zip(members, outs, *seen[0]):
        assert st == 0 and ad == zlib.adler32(m) and zlib.decompress(out) == m.tobytes()


@pytest.mark.parametrize("sizes_known", [True, False])
def test_inflate_batch(ctx, members, sizes_known):
    n = len(members)
    streams = [np.frombuffer(zlib.compress(m.tobytes(), 1)[2:-4], dtype=np.uint8) for m in members]
    ptrs, lens = zd.Context._ptr_arrays(streams)
    mo = np.array([m.size if sizes_known else _lib.SIZE_UNKNOWN for m in members], dtype=np.uint64)
    seen = []

    def call(dst, cap, need, off, ln):
        ck = np.zeros(n, dtype=np.uint32)
        st = np.full(n, -1, dtype=np.int32)
        rc = ctx.L.zipc_b200_inflate_batch(ctx.h, _lib.CK_CRC32, 0, n, ptrs, lens, P(mo, C.c_size_t), dst, cap, need, off, ln,
                                           P(ck, C.c_uint32), P(st, C.c_int))
        seen.append((ck.tolist(), st.tolist()))
        return rc
    outs = arena_twice(ctx, call, n, "inflate_batch")
    assert seen[0] == seen[1]
    for m, out, ck, st in zip(members, outs, *seen[0]):
        assert st == 0 and out == m.tobytes() and ck == zlib.crc32(m)


def test_zlib_decompress_batch(ctx, members):
    n = len(members)
    streams = [np.frombuffer(zlib.compress(m.tobytes(), 1), dtype=np.uint8) for m in members]
    ptrs, lens = zd.Context._ptr_arrays(streams)
    mo = np.array([m.size for m in members], dtype=np.uint64)
    seen = []

    def call(dst, cap, need, off, ln):
        ex = np.zeros(n, dtype=np.uint32)
        fo = np.zeros(n, dtype=np.uint32)
        st = np.full(n, -1, dtype=np.int32)
        rc = ctx.L.zipc_b200_zlib_decompress_batch(ctx.h, _lib.ADLER_RFC1950, n, ptrs, lens, P(mo, C.c_size_t), dst, cap, need, off,
                                                   ln, P(ex, C.c_uint32), P(fo, C.c_uint32), P(st, C.c_int))
        seen.append((ex.tolist(), fo.tolist(), st.tolist()))
        return rc
    outs = arena_twice(ctx, call, n, "zlib_decompress_batch")
    assert seen[0] == seen[1]
    for m, out, ex, fo, st in zip(members, outs, *seen[0]):
        assert st == 0 and out == m.tobytes() and ex == fo == zlib.adler32(m)


def test_zip_extract_batch(ctx, members):
    bio = io.BytesIO()
    with zipfile.ZipFile(bio, "w") as zf:
        for i, m in enumerate(members):  # every fifth member stored, the others deflated
            zf.writestr(zipfile.ZipInfo("m/%02d" % i), m.tobytes(), zipfile.ZIP_STORED if i % 5 == 0 else zipfile.ZIP_DEFLATED, 1)
    archive = np.frombuffer(bio.getvalue(), dtype=np.uint8)
    L = ctx.L
    ms, cnt = C.POINTER(_lib.Member)(), C.c_size_t()
    ctx._check(L.zipc_b200_zip_parse(archive.ctypes.data, archive.size, C.byref(ms), C.byref(cnt)), "zip_parse")
    n = cnt.value
    assert n == len(members)
    seen = []
    try:
        def call(dst, cap, need, off, ln):
            fo = np.zeros(n, dtype=np.uint32)
            st = np.full(n, -1, dtype=np.int32)
            rc = L.zipc_b200_zip_extract_batch(ctx.h, ms, n, dst, cap, need, off, ln, P(fo, C.c_uint32), P(st, C.c_int))
            seen.append((fo.tolist(), st.tolist()))
            return rc
        outs = arena_twice(ctx, call, n, "zip_extract_batch")
    finally:
        L.zipc_b200_free(ms)
    assert seen[0] == seen[1]
    for m, out, fo, st in zip(members, outs, *seen[0]):
        assert st == 0 and out == m.tobytes() and fo == zlib.crc32(m)


# ---- one stream in segments ---------------------------------------------------------------------------------------------
SEG = 256 * KiB


@pytest.fixture(scope="module")
def stream_input(members):
    return np.concatenate(members[:40])


def deflate_segments_twice(ctx, data, primed):
    """(stream, index, crc32) of both runs: without an arena then fetch, and into a pageable arena of the size asked for"""
    fn = ctx.L.zipc_b200_deflate_primed if primed else ctx.L.zipc_b200_deflate_segmented
    nmax = -(-data.size // SEG) + 1
    runs = []
    for with_arena in (False, True):
        index = np.zeros((nmax + 1, 2), dtype=np.uint64)
        dlen, nseg, crc = C.c_size_t(), C.c_size_t(), C.c_uint32(0xDEADBEEF)
        if with_arena:
            out = np.full(runs[0][0].size, 0x5A, dtype=np.uint8)
            rc = fn(ctx.h, _lib.LEVEL_DEFAULT, data.ctypes.data, data.size, SEG, 1, out.ctypes.data, out.size, C.byref(dlen),
                    P(index, C.c_uint64), nmax + 1, C.byref(nseg), C.byref(crc))
            assert rc == _lib.OK
        else:
            rc = fn(ctx.h, _lib.LEVEL_DEFAULT, data.ctypes.data, data.size, SEG, 1, None, 0, C.byref(dlen),
                    P(index, C.c_uint64), nmax + 1, C.byref(nseg), C.byref(crc))
            assert rc == _lib.ERR_DST_TOO_SMALL
            out = np.full(dlen.value, 0xC3, dtype=np.uint8)
            ctx._check(ctx.L.zipc_b200_fetch(ctx.h, out.ctypes.data, out.size), "fetch")
        assert dlen.value == out.size > ARENA_MIN
        runs.append((out, index[:nseg.value + 1].copy(), crc.value))
    (a, ia, ca), (b, ib, cb) = runs
    assert np.array_equal(a, b) and np.array_equal(ia, ib) and ca == cb
    return a, ia, ca


@pytest.mark.parametrize("primed", [False, True])
def test_deflate_segmented_and_primed(ctx, stream_input, primed):
    out, index, crc = deflate_segments_twice(ctx, stream_input, primed)
    assert crc == zlib.crc32(stream_input)
    assert int(index[-1, 0]) == out.size and int(index[-1, 1]) == stream_input.size
    assert zlib.decompress(out.tobytes(), -15) == stream_input.tobytes()


def test_inflate_segmented(ctx, stream_input):
    stream, index, _ = deflate_segments_twice(ctx, stream_input, False)
    L = ctx.L
    nseg = index.shape[0] - 1
    runs = []
    for with_arena in (False, True):
        dlen, crc, st = C.c_size_t(), C.c_uint32(0xDEADBEEF), C.c_int(-1)
        if with_arena:
            out = np.full(stream_input.size, 0x5A, dtype=np.uint8)
            rc = L.zipc_b200_inflate_segmented(ctx.h, stream.ctypes.data, stream.size, P(index, C.c_uint64), nseg, out.ctypes.data,
                                               out.size, C.byref(dlen), C.byref(crc), C.byref(st))
            assert rc == _lib.OK
        else:
            rc = L.zipc_b200_inflate_segmented(ctx.h, stream.ctypes.data, stream.size, P(index, C.c_uint64), nseg, None, 0,
                                               C.byref(dlen), C.byref(crc), C.byref(st))
            assert rc == _lib.ERR_DST_TOO_SMALL
            out = np.full(dlen.value, 0xC3, dtype=np.uint8)
            ctx._check(L.zipc_b200_fetch(ctx.h, out.ctypes.data, out.size), "fetch")
        runs.append((out, dlen.value, crc.value, st.value))
    (a, na, ca, sa), (b, nb, cb, sb) = runs
    assert na == nb == stream_input.size and ca == cb == zlib.crc32(stream_input) and sa == sb == 0
    assert np.array_equal(a, b) and np.array_equal(a, stream_input)
