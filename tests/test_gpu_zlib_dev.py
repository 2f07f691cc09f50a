"""GPU parity of the device-resident zlib entry points (zipc_b200_zlib_compress_batch_dev, zipc_b200_zlib_decompress_batch_dev)
with the host entry points (zipc_b200_zlib_compress_batch, zipc_b200_zlib_decompress_batch), the oracle and Python's zlib.

The buffers follow test_gpu_device_entry_points: allocated with the library's helpers, canary-filled, read back whole;
inputs at every residue mod 16 with real bytes around them, output slots back to back at odd offsets."""
import ctypes as C
import zlib

import numpy as np
import pytest

from oracle import zipc_oracle as zo
from test_gpu_device_entry_points import DevBuf, HEAD, LEVELS, assert_untouched_outside, slot_layout, source_layout
from zipc_b200 import _lib, synth
from zipc_b200 import zipc_deflate as zd

pytestmark = pytest.mark.gpu

MODES = [_lib.ADLER_REF_COMPAT, _lib.ADLER_RFC1950]


@pytest.fixture(scope="module")
def ctx():
    c = zd.Context(0)
    zd.set_default_context(c)
    yield c
    zd.set_default_context(None)
    c.close()


@pytest.fixture
def dev(ctx):
    bufs = []

    def make(size, seed=0):
        b = DevBuf(ctx, size, seed)
        bufs.append(b)
        return b
    yield make
    for b in bufs:
        b.free()


def _sz(vals):
    return (C.c_size_t * max(len(vals), 1))(*vals)


def compress_dev(ctx, level, mode, src, src_off, src_len, dst, dst_off, cap):
    n = len(src_off)
    dl, ad, st = (C.c_size_t * max(n, 1))(), (C.c_uint32 * max(n, 1))(), (C.c_int * max(n, 1))()
    rc = ctx.L.zipc_b200_zlib_compress_batch_dev(ctx.h, LEVELS[level], mode, n,
                                                 src.p if src else None, _sz(src_off), _sz(src_len),
                                                 dst.p if dst else None, _sz(dst_off), _sz(cap), dl, ad, st)
    return rc, list(dl[:n]), list(ad[:n]), list(st[:n])


def decompress_dev(ctx, mode, src, src_off, src_len, dst, dst_off, max_out):
    """-> rc, dst_len, expect, found, status (expect / found start at 0, as in the host call's Python wrapper)"""
    n = len(src_off)
    dl, ex, fo, st = (C.c_size_t * max(n, 1))(), (C.c_uint32 * max(n, 1))(), (C.c_uint32 * max(n, 1))(), (C.c_int * max(n, 1))()
    rc = ctx.L.zipc_b200_zlib_decompress_batch_dev(ctx.h, mode, n, src.p if src else None, _sz(src_off), _sz(src_len),
                                                   dst.p if dst else None, _sz(dst_off), _sz(max_out), dl, ex, fo, st)
    return rc, list(dl[:n]), list(ex[:n]), list(fo[:n]), list(st[:n])


def _placed_source(dev, items, residues, seed=1):
    offs, size = source_layout([len(d) for d in items], residues)
    src = dev(size, seed=seed)
    for o, d in zip(offs, items):
        src.place(o, d)
    src.upload()
    return src, offs


def _compress_placed(ctx, dev, items, level, mode, residues=None, caps=None):
    """one compress_dev call with inputs at the given residues and slots back to back at odd offsets; checks that nothing
    outside the written ranges changed -> (streams or None, adler, status, dst_len, dst buffer, slot offsets, readback)"""
    residues = [i % 16 for i in range(len(items))] if residues is None else residues
    src, offs = _placed_source(dev, items, residues)
    caps = [ctx.L.zipc_b200_zlib_bound(len(d)) for d in items] if caps is None else caps
    doffs, dsize = slot_layout(caps, HEAD + 1, odd=True)
    dst = dev(dsize, seed=2)
    dst.upload()
    rc, dl, ad, st = compress_dev(ctx, level, mode, src, offs, [len(d) for d in items], dst, doffs, caps)
    assert rc == _lib.OK, (rc, ctx.L.zipc_b200_last_error(ctx.h))
    got = dst.read()
    assert_untouched_outside(dst, got, [(doffs[i], doffs[i] + dl[i]) for i in range(len(items))], f"level {level} mode {mode}")
    assert (src.read() == src.image).all(), "the input buffer changed"
    outs = [got[doffs[i]:doffs[i] + dl[i]].tobytes() if st[i] == _lib.OK else None for i in range(len(items))]
    return outs, ad, st, dl, doffs, caps


# ==== compress ============================================================================================================
def _quirk_corpus():
    """as test_gpu_deflate._quirk_corpus: every 5552-byte chunk of most of these has a mean byte of 115 or more, where the
    reference's Adler-32 differs from RFC 1950; plus text members around the block and tile edges"""
    t = np.frombuffer(synth.text_v1(21, 300000).tobytes(), dtype=np.uint8)
    rnd = synth.rand_v1(22, 250001).tobytes()
    text = synth.text_v1(25, 140000).tobytes()
    return [(t | 0x80).tobytes(), rnd, b"\xff" * 200000 + rnd[:5000] + b"\xff" * 70000,
            (t[:90000] | 0x80).tobytes() + rnd[:70000] + bytes(range(256)) * 300 + b"\xfe" * 65534 + t[:50000].tobytes(),
            bytes(range(256)) * 1000, b"\xff" * 5552, b""] + [text[:n] for n in (1, 2, 2049, 61439, 61441, 65536, 131077)]


def _zlib_accepts(stream, data, adler, mode):
    if mode == _lib.ADLER_REF_COMPAT:
        assert zo.zlib_decompress(stream) == (data, adler)      # (raises on a checksum mismatch)
    else:
        assert zlib.decompress(stream) == data and adler == zlib.adler32(data)


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("level", ["none", "fast", "default", "best"])
def test_zlib_compress_dev_equals_the_host_call(ctx, dev, level, mode):
    """every source residue mod 16, slots back to back at odd offsets; streams and adler[] equal the host call's, and the
    oracle (REF_COMPAT) or zlib (RFC1950) reads them"""
    items = _quirk_corpus()
    host = ctx.zlib_compress_batch(items, level, mode)
    for residues in ([i % 16 for i in range(len(items))], [(5 * i + 3) % 16 for i in range(len(items))]):
        outs, ad, st, dl, _, _ = _compress_placed(ctx, dev, items, level, mode, residues)
        quirk = 0
        for i, d in enumerate(items):
            hst, hout, had = host[i]
            assert st[i] == hst == _lib.OK, i
            assert outs[i] == hout.tobytes() and ad[i] == had, (i, len(d), residues[i])
            assert int.from_bytes(outs[i][-4:], "big") == ad[i]
            _zlib_accepts(outs[i], d, ad[i], mode)
            quirk += ad[i] != zlib.adler32(d)
        assert quirk >= 3 if mode == _lib.ADLER_REF_COMPAT else quirk == 0


def test_zlib_compress_dev_large_members_are_split(ctx, dev, monkeypatch):
    """a 3 MiB text member and a 400 KiB one in a thin batch are cut into primed segments, as by the host call"""
    t = np.frombuffer(synth.text_v1(26, 3 << 20).tobytes(), dtype=np.uint8)
    items = [(t | 0x80).tobytes(), synth.text_v1(27, 400 << 10).tobytes()]
    for level in ("fast", "default"):
        host = ctx.zlib_compress_batch(items, level, _lib.ADLER_REF_COMPAT)
        outs, ad, st, dl, _, _ = _compress_placed(ctx, dev, items, level, _lib.ADLER_REF_COMPAT, [7, 10])
        for i, d in enumerate(items):
            assert st[i] == _lib.OK and outs[i] == host[i][1].tobytes() and ad[i] == host[i][2], i
            _zlib_accepts(outs[i], d, ad[i], _lib.ADLER_REF_COMPAT)
        assert ad[0] != zlib.adler32(items[0])
        monkeypatch.setenv("ZIPC_B200_SPLIT_MIN", str(1 << 40))   # the same members on one CTA each: other streams
        whole = ctx.zlib_compress_batch(items, level, _lib.ADLER_REF_COMPAT)
        monkeypatch.delenv("ZIPC_B200_SPLIT_MIN")
        for i in range(len(items)):
            assert whole[i][1].tobytes() != outs[i], i


def test_zlib_compress_dev_bound_at_the_worst_case(ctx, dev):
    """2 MiB of incompressible data alone: 32 segments of 64 KiB, each with stored blocks and an empty stored block.  A slot
    of zipc_b200_zlib_bound is enough (deflate_bound + 6 is not); one byte short of the real length gives DST_TOO_SMALL with
    the whole slot untouched while the neighbours succeed"""
    big = synth.rand_v1(28, 2 << 20).tobytes()
    L = len(big)
    bound = ctx.L.zipc_b200_zlib_bound(L)
    host = ctx.zlib_compress_batch([big], "default", _lib.ADLER_RFC1950)
    for level in ("fast", "default"):
        outs, ad, st, dl, _, _ = _compress_placed(ctx, dev, [big], level, _lib.ADLER_RFC1950, [3], caps=[bound])
        assert st == [_lib.OK] and dl[0] <= bound
        assert dl[0] > ctx.L.zipc_b200_deflate_bound(L) + 6, (dl[0], bound)
        _zlib_accepts(outs[0], big, ad[0], _lib.ADLER_RFC1950)
        if level == "default":
            assert outs[0] == host[0][1].tobytes()
    # the same member one byte short, between two neighbours (the batch stays thin: the member is split the same way)
    small = [synth.text_v1(29, 70000).tobytes(), synth.text_v1(30, 5000).tobytes()]
    items = [small[0], big, small[1]]
    exact = [len(s) for _, s, _ in ctx.zlib_compress_batch(items, "default", _lib.ADLER_REF_COMPAT)]
    assert exact[1] == dl[0]
    caps = [exact[0], exact[1] - 1, exact[2]]
    outs, ad, st, dl, doffs, _ = _compress_placed(ctx, dev, items, "default", _lib.ADLER_REF_COMPAT, [1, 2, 15], caps=caps)
    assert st == [_lib.OK, _lib.ERR_DST_TOO_SMALL, _lib.OK] and dl[1] == 0 and ad[1] == 0
    for i in (0, 2):
        _zlib_accepts(outs[i], items[i], ad[i], _lib.ADLER_REF_COMPAT)
    # (_compress_placed checked every byte outside [doffs[i], doffs[i] + dl[i]): slot 1 is untouched as a whole)


@pytest.mark.parametrize("level", ["none", "fast", "default", "best"])
def test_zlib_compress_dev_of_nothing(ctx, dev, level):
    """an empty input: the 2-byte header, an empty final block, trailer 00000001"""
    for mode in MODES:
        outs, ad, st, dl, _, _ = _compress_placed(ctx, dev, [b"", b"x"], level, mode, [0, 9])
        (hst, hout, had), _ = ctx.zlib_compress_batch([b"", b"x"], level, mode)
        assert st[0] == _lib.OK and ad[0] == 1 and outs[0] == hout.tobytes()
        assert outs[0][-4:] == b"\x00\x00\x00\x01" and outs[0][:2] == hout.tobytes()[:2]
        assert zo.inflate(outs[0][2:-4]) == b"" and zlib.decompress(outs[0]) == b""


# ==== decompress ==========================================================================================================
def _oracle_zlib(s, cap):
    """(status, bytes, expect, found) of the reference's zlib_decompress, expect / found as the C ABI reports them"""
    try:
        out, found = zo.zlib_decompress(bytes(s), cap)
    except zo.OracleError as e:
        return e.status, b"", e.extra.get("expect", 0), e.extra.get("found", 0)
    return _lib.OK, out, int.from_bytes(s[-4:], "big"), found


def _check_decompress_dev(ctx, dev, streams, caps, mode, residues, datas=None):
    """one dev call against the host call (status, dst_len, expect, found, bytes), the oracle (REF_COMPAT: status and
    bytes) or the known data; slots back to back at odd offsets, nothing written outside [off, off + dst_len) (success),
    [off, off + max_out) (a decoding failure) or at all (a rejected header) -> (status, found)"""
    src, offs = _placed_source(dev, streams, residues, seed=11)
    doffs, dsize = slot_layout(caps, HEAD + 1, odd=True)
    dst = dev(dsize, seed=12)
    dst.upload()
    rc, dl, ex, fo, st = decompress_dev(ctx, mode, src, offs, [len(s) for s in streams], dst, doffs, caps)
    assert rc == _lib.OK, (rc, ctx.L.zipc_b200_last_error(ctx.h))
    got = dst.read()
    header_bad = {_lib.ERR_ZLIB_METHOD, _lib.ERR_ZLIB_WINDOW, _lib.ERR_ZLIB_DICT}
    ranges = []
    for i, s in enumerate(streams):
        rejected = len(s) < 6 or st[i] in header_bad or (st[i] == _lib.ERR_CORRUPTED and (s[0] * 256 + s[1]) % 31)
        if not rejected:
            ranges.append((doffs[i], doffs[i] + (dl[i] if st[i] == _lib.OK or st[i] == _lib.ERR_CHECKSUM else caps[i])))
    assert_untouched_outside(dst, got, ranges, f"mode {mode}")
    for i, (hst, hout, hex_, hfo) in enumerate(ctx.zlib_decompress_batch(streams, caps, mode)):
        assert (st[i], dl[i], ex[i], fo[i]) == (hst, len(hout), hex_, hfo), (i, len(streams[i]))
        if st[i] in (_lib.OK, _lib.ERR_CHECKSUM):
            assert got[doffs[i]:doffs[i] + dl[i]].tobytes() == hout.tobytes(), i
    for i, s in enumerate(streams):
        if mode == _lib.ADLER_REF_COMPAT:
            est, eout, eex, efo = _oracle_zlib(s, caps[i])
            assert st[i] == est, (i, st[i], est)
            if est == _lib.OK:
                assert got[doffs[i]:doffs[i] + dl[i]].tobytes() == eout and (ex[i], fo[i]) == (eex, efo), i
            elif est == _lib.ERR_CHECKSUM:
                assert (ex[i], fo[i]) == (eex, efo), i
        if datas is not None and datas[i] is not None and st[i] == _lib.OK:
            assert got[doffs[i]:doffs[i] + dl[i]].tobytes() == datas[i], i
    assert (src.read() == src.image).all(), "the input buffer changed"
    return st, fo


def _decompress_corpus(ctx):
    """(zlib stream, data): Python's zlib at levels 1, 6, 9; this library's zlib_compress (REF_COMPAT, quirk data); the
    oracle's zlib_compress"""
    quirk = _quirk_corpus()
    text = synth.text_v1(31, 120000).tobytes()
    r = synth.rand_v1(32, 40000).tobytes()
    plain = [text, r, bytes(60000), text[:30000] + r[:20000] + text[:30000], b"abc", b""]
    out = [(zlib.compress(d, lvl), d) for d in plain + quirk[:2] for lvl in (1, 6, 9)]
    for level in ("fast", "default", "best"):
        out += [(zs.tobytes(), d) for d, (st, zs, _) in zip(quirk, ctx.zlib_compress_batch(quirk, level, _lib.ADLER_REF_COMPAT))]
    for d in (text[:50000], quirk[0][:40000], quirk[4], b""):
        out.append((zo.zlib_compress(d, "default")[1], d))
    return out


@pytest.mark.parametrize("mode", MODES)
def test_zlib_decompress_dev_valid_streams(ctx, dev, mode):
    """every source residue mod 16, odd output offsets, max_out exact, exact + 1 and exact - 1, each stream through all
    three in turn"""
    corpus = _decompress_corpus(ctx)
    streams = [s for s, _ in corpus]
    for turn in range(3):
        caps = [(len(d), len(d) + 1, max(0, len(d) - 1))[(i + turn) % 3] for i, (_, d) in enumerate(corpus)]
        st, _ = _check_decompress_dev(ctx, dev, streams, caps, mode, [(i + turn) % 16 for i in range(len(streams))],
                                      [d for _, d in corpus])
        assert _lib.OK in st and _lib.ERR_SIZE_EXCEEDED in st
        if mode == _lib.ADLER_REF_COMPAT:
            assert _lib.ERR_CHECKSUM in st     # (zlib's RFC 1950 trailers on quirk data)


def _with_header(s, cmf, fdict=False):
    """s with its header replaced by CMF = cmf and a FLG whose FCHECK is right"""
    flg = 0x20 if fdict else 0
    flg += (31 - (cmf * 256 + flg) % 31) % 31
    return bytes([cmf, flg]) + s[2:]


@pytest.mark.parametrize("mode", MODES)
def test_zlib_decompress_dev_bad_streams(ctx, dev, mode):
    """one batch of lengths 0-5, a bad FCHECK, methods 7 and 15, CINFO 8, FDICT set, a flipped trailer byte, a corrupt body
    and a size overrun, with good streams in between: every status and found as the host call's, rejected headers
    leave their slots untouched"""
    d = synth.text_v1(33, 30000).tobytes()
    good = zlib.compress(d, 6)
    corrupt = bytearray(good)
    for k in range(40, 60):
        corrupt[k] ^= 0x5A
    flipped = bytearray(good)
    flipped[-2] ^= 0x01
    bad = [good[:n] for n in range(6)]
    bad += [bytes([good[0], good[1] ^ 0x01]) + good[2:], _with_header(good, 0x77), _with_header(good, 0x7F),
            _with_header(good, 0x88), _with_header(good, 0x78, fdict=True), bytes(flipped), bytes(corrupt), good]
    streams, caps = [], []
    for k, s in enumerate(bad):
        streams += [s, zlib.compress(d[k * 1000:], 9)]
        caps += [len(d) - 1 if k == len(bad) - 1 else len(d), len(d) - k * 1000]
    st, fo = _check_decompress_dev(ctx, dev, streams, caps, mode, [(3 * i) % 16 for i in range(len(streams))])
    want = [_lib.ERR_CORRUPTED] * 7 + [_lib.ERR_ZLIB_METHOD] * 2 + [_lib.ERR_ZLIB_WINDOW, _lib.ERR_ZLIB_DICT, _lib.ERR_CHECKSUM]
    assert st[0:24:2] == want
    assert st[24] != _lib.OK and st[26] == _lib.ERR_SIZE_EXCEEDED   # (what a corrupt body gives is the host call's, checked above)
    assert fo[14] == 7 and fo[16] == 15
    if mode == _lib.ADLER_RFC1950:
        assert st[1::2] == [_lib.OK] * len(bad)


def test_zlib_decompress_dev_many_warps(ctx, dev, monkeypatch):
    """a large REF_COMPAT stream of quirk data on the many-warp decoder: the Adler-32 folded over its chunks' blocks"""
    monkeypatch.setenv("ZIPC_B200_PAR_MIN", "65536")
    t = np.frombuffer(synth.text_v1(34, 3 << 20).tobytes(), dtype=np.uint8)
    big = (t | 0x80).tobytes()
    monkeypatch.setenv("ZIPC_B200_SPLIT_MIN", str(1 << 40))     # (one CTA: dynamic blocks all the way)
    (_, zs, ad), = ctx.zlib_compress_batch([big], "default", _lib.ADLER_REF_COMPAT)
    monkeypatch.delenv("ZIPC_B200_SPLIT_MIN")
    zs = zs.tobytes()
    small = zlib.compress(synth.text_v1(35, 9000).tobytes())
    p0 = ctx.parallel_streams
    st, fo = _check_decompress_dev(ctx, dev, [small, zs], [9000, len(big)], _lib.ADLER_REF_COMPAT, [4, 13], [None, big])
    p1 = ctx.parallel_streams
    assert st == [_lib.OK, _lib.OK] and fo[1] == ad != zlib.adler32(big)
    assert p1[0] - p0[0] == 2, (p0, p1)    # (the dev call and the host call)


def test_zlib_decompress_dev_truncated_views(ctx, dev):
    """views (start of S, len(S) - d) of one full stream S with its continuation in place: each result is the host call's
    on the cut bytes, so the trailer is read from the cut's end"""
    data = synth.text_v1(36, 200000).tobytes()
    s = zlib.compress(data, 6)
    L = len(s)
    cuts = sorted({L - k for k in range(0, 12)} | {L // 2, 100, 6, 5})
    src = dev(HEAD + L + 64 + 4096 + 256, seed=41)
    a = src.place(HEAD + 5, s)
    src.upload()
    caps = [len(data)] * len(cuts)
    doffs, dsize = slot_layout(caps, HEAD + 1, odd=True)
    dst = dev(dsize, seed=42)
    dst.upload()
    for mode in MODES:
        rc, dl, ex, fo, st = decompress_dev(ctx, mode, src, [a] * len(cuts), cuts, dst, doffs, caps)
        assert rc == _lib.OK
        host = ctx.zlib_decompress_batch([s[:n] for n in cuts], caps, mode)
        for i, (hst, hout, hex_, hfo) in enumerate(host):
            assert (st[i], dl[i], ex[i], fo[i]) == (hst, len(hout), hex_, hfo), (cuts[i], L)
        assert st[cuts.index(L)] == _lib.OK and st[cuts.index(L - 1)] == _lib.ERR_CHECKSUM
        ok = cuts.index(L)
        assert dst.read()[doffs[ok]:doffs[ok] + dl[ok]].tobytes() == data


def test_zlib_decompress_dev_same_range_new_bytes(ctx, dev, monkeypatch):
    """stream A at p decodes (many warps); the range is overwritten with stream B, padded inside to A's length (the bytes
    between B's final block and its trailer are ignored), and decoded again with the same (p, len): the output is B's"""
    monkeypatch.setenv("ZIPC_B200_PAR_MIN", "65536")
    da = synth.text_v1(37, 2 << 20).tobytes()
    db = synth.text_v1(38, (2 << 20) - 4321).tobytes()
    sa, sb = zlib.compress(da, 6), zlib.compress(db, 9)
    assert len(sb) < len(sa)
    L = len(sa)
    sb = sb[:-4] + bytes(L - len(sb)) + sb[-4:]
    cap = len(da) + 1000
    src = dev(HEAD + L + 64 + 4096 + 256, seed=43)
    p = src.place(HEAD + 6, sa)
    src.upload()
    dst = dev(HEAD + cap + 4096 + 256, seed=44)
    dst.upload()

    def decode(want):
        p0 = ctx.parallel_streams
        rc, dl, ex, fo, st = decompress_dev(ctx, _lib.ADLER_RFC1950, src, [p], [L], dst, [HEAD + 3], [cap])
        assert rc == _lib.OK and st == [_lib.OK] and fo == ex == [zlib.adler32(want)]
        assert ctx.parallel_streams[0] == p0[0] + 1, "not decoded by many warps"
        assert dl[0] == len(want) and dst.read()[HEAD + 3:HEAD + 3 + dl[0]].tobytes() == want

    for between in (False, True):
        src.place(p, sa)
        src.upload()
        decode(da)
        src.place(p, sb)
        src.upload(p, p + L)
        if between:
            assert zd.zlib_decompress(sa, decompressed_size=len(da), adler_mode=_lib.ADLER_RFC1950).get_ok()[0] == da
        decode(db)


# ==== arguments ===========================================================================================================
def test_zlib_dev_arguments(ctx, dev):
    """NULL arrays, a bad level or Adler mode, ZIPC_SIZE_UNKNOWN: ZIPC_ERR_INVALID_ARG before anything is written; n = 0 is
    a no-op"""
    d = synth.text_v1(39, 10000).tobytes()
    zs = zlib.compress(d)
    src = dev(HEAD + len(d) + 64 + 4096 + 256, seed=45)
    o = src.place(HEAD, zs)
    src.upload()
    cap = ctx.L.zipc_b200_zlib_bound(len(d))
    dst = dev(HEAD + cap + 4096 + 256, seed=46)
    dst.upload()
    n = 1
    dl, ad, ex, st = (C.c_size_t * 1)(), (C.c_uint32 * 1)(), (C.c_uint32 * 1)(), (C.c_int * 1)()
    so, sl, do, dc = _sz([o]), _sz([len(zs)]), _sz([HEAD + 1]), _sz([cap])
    full = [ctx.h, _lib.LEVEL_DEFAULT, _lib.ADLER_REF_COMPAT, n, src.p, so, sl, dst.p, do, dc, dl, ad, st]
    for k in (0, 4, 5, 6, 7, 8, 9, 10, 12):
        args = list(full)
        args[k] = None
        assert ctx.L.zipc_b200_zlib_compress_batch_dev(*args) == _lib.ERR_INVALID_ARG, k
    for k, v in ((1, -1), (1, 4), (2, 2)):
        args = list(full)
        args[k] = v
        assert ctx.L.zipc_b200_zlib_compress_batch_dev(*args) == _lib.ERR_INVALID_ARG, (k, v)
    full = [ctx.h, _lib.ADLER_RFC1950, n, src.p, so, sl, dst.p, do, _sz([len(d)]), dl, ad, ex, st]
    for k in (0, 3, 4, 5, 6, 7, 8, 9, 12):
        args = list(full)
        args[k] = None
        assert ctx.L.zipc_b200_zlib_decompress_batch_dev(*args) == _lib.ERR_INVALID_ARG, k
    for k, v in ((1, 2), (8, _sz([_lib.SIZE_UNKNOWN]))):
        args = list(full)
        args[k] = v
        assert ctx.L.zipc_b200_zlib_decompress_batch_dev(*args) == _lib.ERR_INVALID_ARG, k
    assert (dst.read() == dst.canary).all()
    assert compress_dev(ctx, "default", _lib.ADLER_REF_COMPAT, None, [], [], None, [], [])[0] == _lib.OK
    assert decompress_dev(ctx, _lib.ADLER_REF_COMPAT, None, [], [], None, [], [])[0] == _lib.OK
    # expect / found may be NULL, adler may be NULL
    assert ctx.L.zipc_b200_zlib_decompress_batch_dev(ctx.h, _lib.ADLER_RFC1950, 1, src.p, so, sl, dst.p, do, _sz([len(d)]), dl,
                                                     None, None, st) == _lib.OK and st[0] == _lib.OK and dl[0] == len(d)
    assert ctx.L.zipc_b200_zlib_compress_batch_dev(ctx.h, _lib.LEVEL_FAST, _lib.ADLER_RFC1950, 1, src.p, _sz([o]), _sz([len(zs)]),
                                                   dst.p, do, dc, dl, None, st) == _lib.OK and st[0] == _lib.OK
    assert (src.read() == src.image).all()
