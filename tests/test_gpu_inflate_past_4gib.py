"""Inflate outputs past 4 GiB, on both decoders, against the streams of big_output_inputs.py, whose output is a 32 KiB
random prefix tiled (known without decoding them; test_big_output_inputs_cpu.py holds the builders to that):

- expand (2^32 + 69,633 bytes): one fixed block of 2^32 + 36,865 bytes, ~80-fold, always on the one-warp decoder, which
  writes past 2^32 there: matches in [2^32, 2^32 + 32768) (the distance check against a 64-bit position), the fused
  Adler-32 of a block of 4 GiB or more, and the count-only pass of a call without sizes;
- spread (2^32 + 69,633 bytes): dynamic blocks of 4 KiB, decoded by many warps, matches in [2^32, 2^32 + 32768);
- big_block (2^32 + 69,633 bytes): one dynamic block of 2^32 + 4097 bytes, decoded by many warps with that block as one
  chunk.  With Adler-32 the block's output length has to be kept in 64 bits: cut to 32, the block lengths no longer add
  up to the output and the stream falls back to the one-warp decoder (the fallback counter says so);
- expand and spread of 2^32 + 1 bytes, for decompressed_size 2^32 - 1, 2^32 (= total - 1) and 2^32 + 1 (= total).

Entry points: zipc_b200_inflate_batch_dev (the slot at an odd offset between canary bytes; spread also between two small
neighbours, canaries around every input and slot) with CRC-32 and the reference's Adler-32, spread also RFC 1950's;
zipc_b200_inflate_batch from host memory into an arena past 4 GiB, sizes known and unknown; big_block through
zipc_b200_zlib_decompress_batch_dev with the right REF_COMPAT trailer and a wrong RFC 1950 one; spread as the member of a
ZIP64 archive through zip_parse_dev and zip_extract_batch_dev; the refusals of deflate_batch_dev and
zip_deflate_archive_dev for a deflated member of 2^32 bytes.  Outputs are compared on the device in 256 MiB slices, CRC-32
against zlib over host slices (cross-checked with zipc_b200_crc32_combine), Adler-32 against
big_output_inputs.adler32_blocks.  Context.parallel_counters says which decoder answered, and decodes are held to a time
limit.

Not covered here: the segmented and primed stream calls (deflate_segmented / inflate_segmented, deflate_primed) past 4 GiB,
with the host zlib read of a primed stream of that size; RFC 1950 Adler-32 fused on the one-warp decoder past 4 GiB (its
REF_COMPAT form and the RFC 1950 host fold are covered); decompressed_size below the output on big_block (every such cap
sends the stream to the one-warp decoder, as spread's does here)."""
import ctypes as C
import time
import zlib

import numpy as np
import pytest

import big_output_inputs as bo
from zipc_b200 import _lib
from zipc_b200 import zipc_deflate as zd

pytestmark = pytest.mark.gpu

REF, RFC = _lib.ADLER_REF_COMPAT, _lib.ADLER_RFC1950
NEED_FREE = 30 * 10 ** 9
SLICE = 256 << 20
CANARY = 0xA5
DST_AT = 17                              # the output slot starts at an odd offset, canaries before and after it
# (builder, output length): the streams of 2^32 + 1 bytes are for decompressed_size around 2^32
STREAMS = {"expand": ("expand", bo.LEN_LONG), "spread": ("spread", bo.LEN_LONG), "big_block": ("big_block", bo.LEN_LONG),
           "expand_cap": ("expand", bo.LEN_JUST_OVER), "spread_cap": ("spread", bo.LEN_JUST_OVER)}
PARALLEL = {"expand": False, "spread": True, "big_block": True}
# Seconds a call may take.  Measured on one B200 (1000 W): spread 0.1-0.9 s; big_block 40 s, because its large block is one
# speculative chunk and so one warp's work (a fallback would add the one-warp decoder's 40 s to that); expand 30 s.
TIME_LIMIT_S = {"expand": 120.0, "spread": 20.0, "big_block": 70.0}
CRC, ADLER = _lib.CK_CRC32, _lib.CK_ADLER32
ZIP_SIZE = 30                            # ZIPC_ERR_ZIP_SIZE


def _sz(vals):
    return (C.c_size_t * max(len(vals), 1))(*vals)


@pytest.fixture(scope="module")
def ctx():
    import torch
    free, _ = torch.cuda.mem_get_info(0)
    if free < NEED_FREE:
        pytest.skip(f"outputs past 4 GiB need {NEED_FREE / 1e9:.0f} GB of free device memory, {free / 1e9:.1f} GB are free")
    c = zd.Context(0)
    yield c
    c.close()


@pytest.fixture(scope="module")
def ref_slice():
    import torch
    return torch.from_numpy(np.tile(np.frombuffer(bo.prefix(), dtype=np.uint8), SLICE // bo.PERIOD)).cuda()


def _crc_reference(total):
    """zlib.crc32 over host slices, and the same from one slice's CRC by zipc_b200_crc32_combine"""
    crc = bo.expected_crc32(total, SLICE)
    L = _lib.lib()
    whole = zlib.crc32(np.tile(np.frombuffer(bo.prefix(), dtype=np.uint8), SLICE // bo.PERIOD))
    comb = 0
    for off in range(0, total - SLICE + 1, SLICE):
        comb = L.zipc_b200_crc32_combine(comb, whole, SLICE) if off else whole
    rest = total % SLICE
    comb = L.zipc_b200_crc32_combine(comb, zlib.crc32(bo.expected(total, total - rest)), rest)
    assert comb == crc
    return crc


@pytest.fixture(scope="module")
def stream(request, ctx):
    """(Big, device buffer with the stream at byte 3 and other bytes around it, its crc32)"""
    import torch
    name, total = STREAMS[request.param]
    big = bo.BUILDERS[name](total)
    raw = np.frombuffer(bytearray(big.stream()), dtype=np.uint8)
    buf = torch.full((raw.size + 3 + 64,), 0xC3, dtype=torch.uint8, device="cuda:0")
    buf[3:3 + raw.size].copy_(torch.from_numpy(raw))
    torch.cuda.synchronize()
    yield big, raw, buf, _crc_reference(big.total)
    del buf
    torch.cuda.empty_cache()


@pytest.fixture(scope="module")
def out_slot(ctx):
    import torch
    n = bo.LEN_LONG + DST_AT + 64
    dst = torch.empty(n, dtype=torch.uint8, device="cuda:0")
    yield dst
    del dst
    torch.cuda.empty_cache()


def _inflate_dev(ctx, buf, n_src, dst, cap, ck, mode):
    dl, cs, st = (C.c_size_t * 1)(), (C.c_uint32 * 1)(), (C.c_int * 1)()
    rc = ctx.L.zipc_b200_inflate_batch_dev(ctx.h, ck, mode, 1, buf.data_ptr(), _sz([3]), _sz([n_src]), dst.data_ptr(),
                                           _sz([DST_AT]), _sz([cap]), dl, cs, st)
    assert rc == _lib.OK
    return st[0], dl[0], cs[0]


def _same_output(dst, at, total, ref_slice):
    for k in range(0, total, SLICE):
        m = min(SLICE, total - k)
        assert bool((dst[at + k:at + k + m] == ref_slice[:m]).all()), f"output differs in [{k}, {k + m})"


def _canaries_intact(dst, total):
    assert bool((dst[:DST_AT] == CANARY).all()) and bool((dst[DST_AT + total:] == CANARY).all())


def _counted(ctx, before, name, calls=1):
    d = [a - b for a, b in zip(ctx.parallel_counters, before)]
    assert d[:2] == ([calls, 0] if PARALLEL[name] else [0, calls]), f"{name}: parallel / fallback moved by {d[:2]}"


# (a call of expand or big_block takes 30-40 s, so RFC 1950 runs on spread here and on big_block in test_zlib_dev_trailers)
@pytest.mark.parametrize("stream,ck,mode", [("expand", CRC, REF), ("expand", ADLER, REF), ("spread", CRC, REF),
                                            ("spread", ADLER, REF), ("spread", ADLER, RFC), ("big_block", CRC, REF),
                                            ("big_block", ADLER, REF)],
                         ids=["expand-crc32", "expand-adler32_ref", "spread-crc32", "spread-adler32_ref", "spread-adler32_rfc",
                              "big_block-crc32", "big_block-adler32_ref"], indirect=["stream"])
def test_inflate_dev(ctx, stream, out_slot, ref_slice, ck, mode):
    big, raw, buf, crc = stream
    name, total = big.name, big.total
    out_slot.fill_(CANARY)
    before = ctx.parallel_counters
    t0 = time.perf_counter()
    st, dl, cs = _inflate_dev(ctx, buf, raw.size, out_slot, total, ck, mode)
    took = time.perf_counter() - t0
    print(f"{name} {total} ck={ck} mode={mode}: {took:.2f} s")
    assert (st, dl) == (_lib.OK, total)
    _counted(ctx, before, name)
    assert took < TIME_LIMIT_S[name]
    want = crc if ck == _lib.CK_CRC32 else bo.adler32_blocks(big, "ref" if mode == REF else "rfc")
    assert cs == want
    _same_output(out_slot, DST_AT, total, ref_slice)
    _canaries_intact(out_slot, total)


@pytest.mark.parametrize("stream,caps", [("expand_cap", [(1 << 32) - 1, 1 << 32, (1 << 32) + 1]),
                                         ("spread_cap", [1 << 32, (1 << 32) + 1])], ids=["one_warp", "many_warps"],
                         indirect=["stream"])
def test_decompressed_size_around_2_32(ctx, stream, out_slot, ref_slice, caps):
    """streams of 2^32 + 1 bytes: decompressed_size 2^32 - 1 and 2^32 (= total - 1) are exceeded, 2^32 + 1 (= total) is
    not, the reference's rule (output > cap); nothing is written past the cap.  The many-warp decoder sees the plan's
    total over the cap and leaves the stream to the one-warp decoder, which reports it (a fallback); at the total it
    decodes the stream itself"""
    big, raw, buf, crc = stream
    for cap in caps:
        out_slot.fill_(CANARY)
        before = ctx.parallel_counters
        t0 = time.perf_counter()
        st, dl, cs = _inflate_dev(ctx, buf, raw.size, out_slot, cap, CRC, REF)
        print(f"{big.name} cap {cap}: {time.perf_counter() - t0:.2f} s")
        d = [a - b for a, b in zip(ctx.parallel_counters, before)]
        assert bool((out_slot[:DST_AT] == CANARY).all()) and bool((out_slot[DST_AT + cap:] == CANARY).all())
        if cap < big.total:
            assert (st, dl, cs) == (_lib.ERR_SIZE_EXCEEDED, 0, 0)
            assert d[:2] == [0, 1]
        else:
            assert (st, dl, cs) == (_lib.OK, big.total, crc)
            assert d[:2] == ([1, 0] if PARALLEL[big.name] else [0, 1])
            _same_output(out_slot, DST_AT, big.total, ref_slice)


@pytest.mark.parametrize("stream", ["spread"], indirect=True)
def test_inflate_dev_between_neighbours(ctx, stream):
    """spread in a batch between two small streams, every input and every output slot with canary bytes around it; the
    large stream is decoded by many warps, the small ones by one warp each"""
    import torch
    big, raw, buf, crc = stream
    small = [bytes(range(256)) * 37 + b"first", b"last neighbour " * 501]
    comp = [np.frombuffer(zlib.compress(x)[2:-4], dtype=np.uint8) for x in small]
    gap = 29
    src_off = [gap, gap + comp[0].size + gap, gap + comp[0].size + gap + raw.size + gap]
    src = torch.full((src_off[2] + comp[1].size + gap,), 0xC3, dtype=torch.uint8, device="cuda:0")
    for o, x in zip(src_off, [comp[0], raw, comp[1]]):
        src[o:o + x.size].copy_(torch.from_numpy(x.copy()))
    caps = [len(small[0]), big.total, len(small[1])]
    dst_off = [gap, gap + caps[0] + gap, gap + caps[0] + gap + caps[1] + gap]
    dst = torch.full((dst_off[2] + caps[2] + gap,), CANARY, dtype=torch.uint8, device="cuda:0")
    dl, cs, st = (C.c_size_t * 3)(), (C.c_uint32 * 3)(), (C.c_int * 3)()
    before = ctx.parallel_counters
    src_len = [comp[0].size, raw.size, comp[1].size]
    assert ctx.L.zipc_b200_inflate_batch_dev(ctx.h, CRC, REF, 3, src.data_ptr(), _sz(src_off), _sz(src_len), dst.data_ptr(),
                                             _sz(dst_off), _sz(caps), dl, cs, st) == _lib.OK
    _counted(ctx, before, big.name)
    assert list(st) == [_lib.OK] * 3 and list(dl) == caps
    assert list(cs) == [zlib.crc32(small[0]), crc, zlib.crc32(small[1])]
    assert bytes(dst[dst_off[0]:dst_off[0] + caps[0]].cpu().numpy()) == small[0]
    assert bytes(dst[dst_off[2]:dst_off[2] + caps[2]].cpu().numpy()) == small[1]
    ref = torch.from_numpy(np.tile(np.frombuffer(bo.prefix(), dtype=np.uint8), SLICE // bo.PERIOD)).cuda()
    _same_output(dst, dst_off[1], big.total, ref)
    for lo, hi in [(0, dst_off[0]), (dst_off[0] + caps[0], dst_off[1]), (dst_off[1] + caps[1], dst_off[2]),
                   (dst_off[2] + caps[2], dst.numel())]:
        assert hi - lo == gap and bool((dst[lo:hi] == CANARY).all())
    del src, dst, ref
    torch.cuda.empty_cache()


@pytest.mark.parametrize("stream", ["spread"], indirect=True)
def test_zip64_member_extract_dev(ctx, stream, out_slot, ref_slice):
    """spread as the deflated member of a ZIP64 archive built by hand (big_output_inputs.zip64_archive; CPython's zipfile
    reads it, test_big_output_inputs_cpu.py), in device memory at an odd offset: zip_parse_dev with ZIP64 allowed, then
    zip_extract_batch_dev, decoded by many warps and checked against the member's CRC-32"""
    import torch
    from zipc_b200 import zipc
    big, raw, buf, crc = stream
    arc, at = bo.zip64_archive(bytes(raw), big.total, crc)
    d = torch.full((len(arc) + 2,), 0xC3, dtype=torch.uint8, device="cuda:0")
    d[1:1 + len(arc)].copy_(torch.from_numpy(np.frombuffer(arc, dtype=np.uint8).copy()))
    mp, cnt = C.POINTER(_lib.Member)(), C.c_size_t()
    assert ctx.L.zipc_b200_zip_parse_dev(ctx.h, d.data_ptr() + 1, len(arc), zipc.ZIP_ALLOW_ZIP64, C.byref(mp),
                                         C.byref(cnt)) == _lib.OK
    try:
        assert cnt.value == 1 and C.string_at(mp[0].path, mp[0].path_len) == bo.ZIP_NAME
        assert (mp[0].compression, mp[0].compressed_size, mp[0].decompressed_size, mp[0].crc32) == (8, raw.size, big.total, crc)
        out_slot.fill_(CANARY)
        dl, fo, st = (C.c_size_t * 1)(), (C.c_uint32 * 1)(), (C.c_int * 1)()
        before = ctx.parallel_counters
        assert ctx.L.zipc_b200_zip_extract_batch_dev(ctx.h, mp, 1, out_slot.data_ptr(), _sz([DST_AT]), dl, fo, st) == _lib.OK
    finally:
        ctx.L.zipc_b200_free(C.cast(mp, C.c_void_p))
    _counted(ctx, before, big.name)
    assert (st[0], dl[0], fo[0]) == (_lib.OK, big.total, crc)
    _same_output(out_slot, DST_AT, big.total, ref_slice)
    _canaries_intact(out_slot, big.total)
    del d


def test_refusals_at_4_gib(ctx, out_slot):
    """a member of 2^32 bytes: deflate_batch_dev refuses it (ZIPC_ERR_INVALID_ARG), zip_deflate_archive_dev refuses it
    deflated (ZIPC_ERR_ZIP_SIZE), both before anything runs; a stored member that size is accepted
    (test_gpu_checksum_edges.py::test_stored_member_past_4_gib)"""
    import torch
    n = 1 << 32
    small = torch.zeros(4096, dtype=torch.uint8, device="cuda:0")
    dl, cs, st = (C.c_size_t * 1)(), (C.c_uint32 * 1)(), (C.c_int * 1)()
    assert ctx.L.zipc_b200_deflate_batch_dev(ctx.h, _lib.LEVEL_DEFAULT, CRC, REF, 1, out_slot.data_ptr(), _sz([0]), _sz([n]),
                                             small.data_ptr(), _sz([0]), _sz([small.numel()]), dl, cs, st) == _lib.ERR_INVALID_ARG
    path = b"big.bin"
    pp, pl = (C.c_void_p * 1)(C.cast(C.c_char_p(path), C.c_void_p).value), (C.c_uint32 * 1)(len(path))
    out_len = C.c_size_t()
    from zipc_b200 import zipc
    assert ctx.L.zipc_b200_zip_deflate_archive_dev(ctx.h, _lib.LEVEL_DEFAULT, 1, pp, pl, out_slot.data_ptr(), _sz([0]), _sz([n]),
                                                   (C.c_int32 * 1)(8), None, None, None, zipc.ZIP_ALLOW_ZIP64,
                                                   small.data_ptr(), small.numel(), C.byref(out_len)) == ZIP_SIZE


@pytest.mark.parametrize("stream,known", [("spread", True), ("spread", False), ("expand", False)],
                         ids=["spread-size_known", "spread-size_unknown", "expand-size_unknown"], indirect=["stream"])
def test_inflate_host_arena_past_4_gib(ctx, stream, known):
    """from host memory, a small stream behind it: the arena is laid out past 4 GiB (dst_need, dst_off); without sizes,
    a count-only pass sizes the outputs first (expand: on one warp)"""
    big, raw, buf, crc = stream
    small = np.frombuffer(zlib.compress(b"tail of the arena " * 100)[2:-4], dtype=np.uint8).copy()
    small_out = b"tail of the arena " * 100
    items = [raw, small]
    ptrs = (C.c_void_p * 2)(*(x.ctypes.data for x in items))
    lens = _sz([raw.size, small.size])
    mo = _sz([big.total, len(small_out)] if known else [_lib.SIZE_UNKNOWN, _lib.SIZE_UNKNOWN])
    need, off, ln = C.c_size_t(), (C.c_size_t * 2)(), (C.c_size_t * 2)()
    ck, stt = (C.c_uint32 * 2)(), (C.c_int * 2)()
    before = ctx.parallel_counters
    rc = ctx.L.zipc_b200_inflate_batch(ctx.h, _lib.CK_CRC32, REF, 2, ptrs, lens, mo, None, 0, C.byref(need), off, ln, ck, stt)
    assert rc == _lib.ERR_DST_TOO_SMALL and need.value >= big.total + len(small_out)
    arena = np.empty(need.value, dtype=np.uint8)
    assert ctx.L.zipc_b200_fetch(ctx.h, arena.ctypes.data, arena.size) == _lib.OK
    _counted(ctx, before, big.name, 1 if known else 2)   # (unknown: the sizing pass, then the real pass from its plan)
    assert list(stt) == [_lib.OK, _lib.OK] and list(ln) == [big.total, len(small_out)]
    assert list(ck) == [crc, zlib.crc32(small_out)]
    assert off[1] >= off[0] + big.total > 1 << 32
    assert arena[off[1]:off[1] + ln[1]].tobytes() == small_out
    for k in range(0, big.total, SLICE):
        m = min(SLICE, big.total - k)
        assert np.array_equal(arena[off[0] + k:off[0] + k + m], bo.expected(big.total, k, m)), k


@pytest.mark.parametrize("stream", ["big_block"], indirect=True)
def test_zlib_dev_trailers(ctx, stream, out_slot, ref_slice):
    """big_block as a zlib stream: the trailer is the block fold, REF_COMPAT with the right trailer; RFC 1950 with a wrong
    one is ZIPC_ERR_CHECKSUM with found = the fold"""
    import torch
    big, raw, buf, crc = stream
    z = torch.empty(raw.size + 6 + 8, dtype=torch.uint8, device="cuda:0")
    z[1:3].copy_(torch.tensor([0x78, 0x9C], dtype=torch.uint8))
    z[3:3 + raw.size].copy_(buf[3:3 + raw.size])
    for mode, wrong in [(REF, False), (RFC, True)]:
        want = bo.adler32_blocks(big, "ref" if mode == REF else "rfc")
        trailer = want ^ 1 if wrong else want
        z[3 + raw.size:7 + raw.size].copy_(torch.tensor(list(trailer.to_bytes(4, "big")), dtype=torch.uint8))
        out_slot.fill_(CANARY)
        dl, ex, fo, st = (C.c_size_t * 1)(), (C.c_uint32 * 1)(), (C.c_uint32 * 1)(), (C.c_int * 1)()
        before = ctx.parallel_counters
        t0 = time.perf_counter()
        assert ctx.L.zipc_b200_zlib_decompress_batch_dev(ctx.h, mode, 1, z.data_ptr(), _sz([1]), _sz([raw.size + 6]),
                                                         out_slot.data_ptr(), _sz([DST_AT]), _sz([big.total]), dl, ex, fo,
                                                         st) == _lib.OK
        took = time.perf_counter() - t0
        _counted(ctx, before, big.name)
        assert took < TIME_LIMIT_S[big.name]
        assert (ex[0], fo[0]) == (trailer, want)
        assert st[0] == (_lib.ERR_CHECKSUM if wrong else _lib.OK)
        if not wrong:
            assert dl[0] == big.total
    _same_output(out_slot, DST_AT, big.total, ref_slice)
    del z
