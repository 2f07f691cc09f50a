"""CRC-32 and Adler-32 kernels at their tile, chain and 4 GiB boundaries, against zlib, the oracle and the chunk model of
checksum_inputs.py (whose layouts test_checksum_inputs_cpu.py holds to their plans).

  1. adler_fold_kernel (reference flavour) on inputs built chunk by chunk: U chunks first and last in a tile, tiles headed by
     low-W chunks behind a negative or non-negative state (they wait on the chain), whole tiles of them, input lengths at
     and around whole tiles, first chunks of 1, 5551 and 5552 bytes; adler_reduce_rfc_kernel at the edges of its CTAs.
  2. The chain between calls on one context: tile counts that go up and down, a context that regrows its chain, two
     contexts on one device taking turns.
  3. crc32_combine_tiles_kernel: full-tile counts F at multiples of 1024 G and around them, every kind of last tile, and the
     length at which the tile grows from 4 KiB.
  4. Past 4 GiB: crc32_dev / adler32_dev, and a stored member whose tiles have 2^32 bytes or more after them, through
     zip_extract_batch_dev and zip_deflate_archive_dev.

Not covered: the wrap of the Adler chain's epoch counter (after 2^32 launches on one context).  Inflate outputs over 4 GiB
are in test_gpu_inflate_past_4gib.py."""
import ctypes as C
import zlib

import numpy as np
import pytest

import checksum_inputs as ci
from oracle import zipc_oracle as zo
from zipc_b200 import _lib, zipc
from zipc_b200 import zipc_deflate as zd

pytestmark = pytest.mark.gpu

REF, RFC = _lib.ADLER_REF_COMPAT, _lib.ADLER_RFC1950


@pytest.fixture(scope="module")
def ctx():
    c = zd.Context(0)
    zd.set_default_context(c)
    yield c
    zd.set_default_context(None)
    c.close()


def _adler_dev(ctx, p, n, mode):
    out = C.c_uint32()
    ctx._check(ctx.L.zipc_b200_adler32_dev(ctx.h, p, n, mode, C.byref(out)), "adler32_dev")
    return out.value


def _crc_dev(ctx, p, n):
    out = C.c_uint32()
    ctx._check(ctx.L.zipc_b200_crc32_dev(ctx.h, p, n, C.byref(out)), "crc32_dev")
    return out.value


def _on_device(host, residue):
    """host bytes at byte `residue` of a device buffer, with other bytes before and after them"""
    import torch
    buf = torch.full((host.size + residue + 64,), 0xA7, dtype=torch.uint8, device="cuda:0")
    buf[residue:residue + host.size].copy_(torch.from_numpy(host))
    torch.cuda.synchronize()
    return buf


# ==== 1. the Adler-32 fold ==================================================================================================
@pytest.mark.parametrize("name", list(ci.LAYOUTS))
def test_adler32_layouts(ctx, name):
    inp = ci.layout(name)
    b = inp.data.tobytes()
    ref, rfc = zo.adler32(b), zlib.adler32(b)
    assert ci.model(inp.data)[0] == ref
    assert ctx.adler32(inp.data, REF) == ref
    assert ctx.adler32(inp.data, RFC) == rfc
    buf = _on_device(inp.data, 7)
    assert _adler_dev(ctx, buf.data_ptr() + 7, inp.data.size, REF) == ref
    assert _adler_dev(ctx, buf.data_ptr() + 7, inp.data.size, RFC) == rfc


def test_adler32_rfc_reduce_cta_edges(ctx):
    """nchunks = m 8192 + {-1, 0, 1}: the last CTA of adler_reduce_rfc_kernel full, one chunk short, or holding one chunk"""
    rng = np.random.default_rng(8)
    top = 3 * ci.RED + 1
    for fill in ("random", 0xFF):
        data = np.frombuffer(rng.bytes(top * ci.CHUNK), dtype=np.uint8) if fill == "random" else \
            np.full(top * ci.CHUNK, 0xFF, dtype=np.uint8)
        for m in (1, 2, 3):
            for d in (-1, 0, 1):
                for first in (1, 5552):
                    v = data[:first + (m * ci.RED + d - 1) * ci.CHUNK]
                    assert ci.chunk_grid(v.size) == (first, m * ci.RED + d)
                    assert ctx.adler32(v, RFC) == zlib.adler32(v), (fill, m, d, first)
                    assert ctx.adler32(v, REF) == zo.adler32(v.tobytes()), (fill, m, d, first)


# ==== 2. the chain between calls ============================================================================================
def _quirk_zlib_round(ctx):
    data = b"\xff" * 300_000 + bytes(range(256)) * 400
    adler, stream = zo.zlib_compress(data, "default")
    [(st, out, expect, found)] = ctx.zlib_decompress_batch([stream])
    assert st == _lib.OK and out.tobytes() == data and expect == found == adler


def test_adler32_chain_reuse(ctx):
    """Tags keep a call from reading what an earlier call left in the chain: calls of 5, 2, 5, 1 and 3 tiles in a row, with
    RFC calls and a zlib_decompress between them; a fresh context that regrows its chain (1, 6, 2 tiles); two contexts
    taking turns.  Every tile of these inputs after the first waits on its predecessor's state."""
    ins = {"a": ci.chained(6, 1), "b": ci.chained(6, 2)}
    refs = {}

    def check(c, which, k):
        v = ci.prefix(ins[which], k)
        if (which, k) not in refs:
            refs[which, k] = zo.adler32(v.tobytes())
        assert c.adler32(v, REF) == refs[which, k], (which, k)

    small = np.frombuffer(np.random.default_rng(9).bytes(3_000_017), dtype=np.uint8)
    for i, (which, k) in enumerate([("a", 5), ("b", 2), ("b", 5), ("a", 1), ("b", 3)]):
        check(ctx, which, k)
        assert ctx.adler32(small[i:], RFC) == zlib.adler32(small[i:])
        _quirk_zlib_round(ctx)
    fresh = zd.Context(0)
    try:
        for which, k in [("a", 1), ("b", 6), ("a", 2)]:
            check(fresh, which, k)
        for c, which, k in [(ctx, "a", 3), (fresh, "b", 5), (ctx, "b", 2), (fresh, "a", 1), (ctx, "a", 6), (fresh, "b", 2),
                            (ctx, "b", 6), (fresh, "a", 4)]:
            check(c, which, k)
    finally:
        fresh.close()


# ==== 3. the CRC-32 tile combine ============================================================================================
def _sm_count():
    import torch
    return torch.cuda.get_device_properties(0).multi_processor_count


def _crc_tile(n, knob, sms):
    """crc32_launch_buffer's tile length for n bytes (restated to say which case a length is)"""
    tile = max(-(-n // (sms * 32)), 4096)
    if knob is not None and 4096 <= knob < tile:
        tile = knob
    return (tile + 511) & ~511


def _crc_three_ways(ctx, host, dev, word, n):
    """crc32 (host bytes), crc32_dev and crc32_dev_async of the first n bytes, against zlib"""
    want = zlib.crc32(host[:n])
    assert ctx.crc32(host[:n]) == want, n
    assert _crc_dev(ctx, dev.data_ptr() + 3, n) == want, n
    ctx._check(ctx.L.zipc_b200_crc32_dev_async(ctx.h, dev.data_ptr() + 3, n, word.data_ptr()), "crc32_dev_async")
    ctx._check(ctx.L.zipc_b200_sync(ctx.h), "sync")
    assert int(word.item()) & 0xFFFFFFFF == want, n


def test_crc32_combine_edges(ctx, monkeypatch):
    """F full tiles and a last tile of last_len bytes, tiles of 4096 and 4608 bytes set with ZIPC_B200_CRC_TILE: F at and
    around 1024 G (G = tiles per thread of the combine, 1 to 17), last_len from 1 byte to a whole tile"""
    import torch
    sms = _sm_count()
    top = 16385 * 4608 + 4608
    host = np.frombuffer(bytearray(np.random.default_rng(10).bytes(top)), dtype=np.uint8)
    dev = _on_device(host, 3)
    word = torch.zeros(1, dtype=torch.int32, device="cuda:0")
    seen = set()
    for knob, Fs in ((4096, (1023, 1024, 1025, 2047, 2048, 2049, 16383, 16384, 16385)), (4608, (16383, 16384, 16385))):
        monkeypatch.setenv("ZIPC_B200_CRC_TILE", str(knob))
        for F in Fs:
            for last in (1, 15, 16, 511, 512, 513, knob - 1, knob):
                n = F * knob + last
                assert _crc_tile(n, knob, sms) == knob, (knob, F, last)
                _crc_three_ways(ctx, host, dev, word, n)
                seen.add(-(-F // 1024))
    assert seen == {1, 2, 3, 16, 17}
    monkeypatch.delenv("ZIPC_B200_CRC_TILE")
    edge = sms * 32 * 4096          # above this the tile grows from 4 KiB (4736 tiles on 148 SMs)
    host = np.frombuffer(bytearray(np.random.default_rng(11).bytes(edge + 512)), dtype=np.uint8)
    dev = _on_device(host, 3)
    for d in (-1, 0, 1, 512):
        assert _crc_tile(edge + d, None, sms) == (4096 if d <= 0 else 4608)
        _crc_three_ways(ctx, host, dev, word, edge + d)


# ==== 4. past 4 GiB =========================================================================================================
PATTERN = 1_000_003                  # a prime: a wrong offset at 2^32, or at a multiple of a tile, reads other bytes
STORED_AT = 3
STORED_LEN = (1 << 32) + (256 << 10) + 4097   # its first 256 KiB tile has 2^32 + 4097 bytes after it
BIG = STORED_AT + STORED_LEN
NEED_FREE = 14 * 10 ** 9


def _pattern():
    return np.frombuffer(bytearray(np.random.default_rng(41).bytes(PATTERN)), dtype=np.uint8)


def _pieces(pat2, start, n, first):
    """the n bytes from offset start of the repeated pattern, as a first piece of `first` bytes and then pieces of
    180 * 5552 bytes; pat2 is the pattern twice"""
    step = 180 * ci.CHUNK
    off, size = 0, first
    while off < n:
        size = min(size, n - off)
        p = (start + off) % PATTERN
        yield pat2[p:p + size]
        off += size
        size = step


def _references(pat2, start, n):
    """(crc32, reference-flavour Adler-32, RFC 1950 Adler-32) of n bytes of the repeated pattern, piece by piece.  The
    reference's word depends on the chunk grid of the whole buffer, so its pieces are the first chunk (len mod 5552 bytes),
    then whole chunks, folded by the chunk model with the signed s2 carried from piece to piece.  (zo.adler32_update
    cannot carry it: the state it takes is packed, and a negative s2 does not survive the packing.)"""
    crc, rfc = 0, 1
    for piece in _pieces(pat2, start, n, 180 * ci.CHUNK):
        crc, rfc = zlib.crc32(piece, crc), zlib.adler32(piece, rfc)
    s1, s2 = 1, 0
    for piece in _pieces(pat2, start, n, ci.chunk_grid(n)[0]):
        for k, a, b in zip(*(x.tolist() for x in ci.chunk_sums(piece))):
            s1, s2, _ = ci.step(s1, s2, k, a, b)
    return crc, ci.pack(s1, s2), rfc


@pytest.fixture(scope="module")
def big(ctx):
    """the pattern repeated over BIG bytes of device memory (byte i = pattern[i mod PATTERN]), built on the device"""
    import torch
    free, _ = torch.cuda.mem_get_info(0)
    if free < NEED_FREE:
        pytest.skip(f"the 4 GiB cases need {NEED_FREE / 1e9:.0f} GB of free device memory, {free / 1e9:.1f} GB are free")
    pat = _pattern()
    buf = torch.empty(BIG, dtype=torch.uint8, device="cuda:0")
    buf[:PATTERN].copy_(torch.from_numpy(pat))
    k = PATTERN
    while k < BIG:
        m = min(k, BIG - k)
        buf[k:k + m].copy_(buf[:m])
        k += m
    torch.cuda.synchronize()
    yield buf, np.concatenate([pat, pat])
    del buf
    torch.cuda.empty_cache()


@pytest.mark.parametrize("n", [(1 << 32) - 1, 1 << 32, (1 << 32) + (256 << 10) + 3])
def test_checksums_past_4_gib(ctx, big, n):
    buf, pat2 = big
    assert int(buf[n - 1]) == int(pat2[(n - 1) % PATTERN])
    crc, ref, rfc = _references(pat2, 0, n)
    assert _crc_dev(ctx, buf.data_ptr(), n) == crc
    assert _adler_dev(ctx, buf.data_ptr(), n, REF) == ref
    assert _adler_dev(ctx, buf.data_ptr(), n, RFC) == rfc


def test_stored_member_past_4_gib(ctx, big):
    """a stored member of 2^32 + 256 KiB + 4097 bytes built by the caller, through zip_extract_batch_dev (copy and CRC in one
    pass, tiles with 2^32 bytes or more after them), then as the only stored member of zip_deflate_archive_dev with ZIP64
    allowed, its directory read back by zip_parse_dev"""
    import torch
    buf, pat2 = big
    crc = 0
    for piece in _pieces(pat2, STORED_AT, STORED_LEN, 180 * ci.CHUNK):
        crc = zlib.crc32(piece, crc)
    L, h = ctx.L, ctx.h
    m = _lib.Member()
    m.compression, m.compressed_bytes, m.start = 0, buf.data_ptr(), STORED_AT
    m.compressed_size = m.decompressed_size = STORED_LEN
    m.crc32 = crc
    dst = torch.empty(STORED_LEN + 1, dtype=torch.uint8, device="cuda:0")
    dl, fo, st = (C.c_size_t * 1)(), (C.c_uint32 * 1)(), (C.c_int * 1)()
    one = (_lib.Member * 1)(m)
    assert L.zipc_b200_zip_extract_batch_dev(h, one, 1, dst.data_ptr(), (C.c_size_t * 1)(1), dl, fo, st) == _lib.OK
    assert (st[0], dl[0], fo[0]) == (_lib.OK, STORED_LEN, crc)
    assert bool(torch.equal(dst[1:], buf[STORED_AT:STORED_AT + STORED_LEN]))
    del dst
    torch.cuda.empty_cache()
    # the archive writer: the member's CRC-32 in its directory entry
    path = b"big.bin"
    pp, pl = (C.c_void_p * 1)(C.cast(C.c_char_p(path), C.c_void_p).value), (C.c_uint32 * 1)(len(path))
    comp = (C.c_int32 * 1)(0)
    lens = (C.c_size_t * 1)(STORED_LEN)
    cap = L.zipc_b200_zip_archive_bound(1, pl, lens, comp)
    out = torch.empty(cap + 1, dtype=torch.uint8, device="cuda:0")
    out_len = C.c_size_t()
    assert L.zipc_b200_zip_deflate_archive_dev(h, _lib.LEVEL_DEFAULT, 1, pp, pl, buf.data_ptr(), (C.c_size_t * 1)(STORED_AT),
                                               lens, comp, None, None, None, zipc.ZIP_ALLOW_ZIP64, out.data_ptr() + 1, cap,
                                               C.byref(out_len)) == _lib.OK
    mp, cnt = C.POINTER(_lib.Member)(), C.c_size_t()
    assert L.zipc_b200_zip_parse_dev(h, out.data_ptr() + 1, out_len.value, zipc.ZIP_ALLOW_ZIP64, C.byref(mp),
                                     C.byref(cnt)) == _lib.OK
    try:
        assert cnt.value == 1 and C.string_at(mp[0].path, mp[0].path_len) == path
        assert (mp[0].compression, mp[0].compressed_size, mp[0].decompressed_size) == (0, STORED_LEN, STORED_LEN)
        assert mp[0].crc32 == crc
    finally:
        L.zipc_b200_free(C.cast(mp, C.c_void_p))
    del out
    torch.cuda.empty_cache()
