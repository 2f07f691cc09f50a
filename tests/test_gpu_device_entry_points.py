"""GPU parity of the device-resident entry points (zipc_b200_deflate_batch_dev, zipc_b200_inflate_batch_dev,
zipc_b200_crc32_dev / _dev_async, zipc_b200_adler32_dev) against the references: the host encoder model and the oracle for
bytes, zlib and the oracle for checksums, the host entry points where the contract is "as the host path".

A caller's device buffers are not the library's arena: inputs sit at any byte offset with real bytes around them (the
continuation of a truncated member, the next member of an archive), output slots sit back to back and need not be
16-byte aligned, and the same device range can be rewritten between two calls.  Every buffer here is allocated with the
library's own helpers, filled with a canary pattern, and read back whole, so a test sees every byte a call changed.  No
access is meant to leave an allocation: inputs start at least HEAD bytes in, and TAIL bytes stay unused after the last
byte a test places or expects to be read."""
import ctypes as C
import zlib

import numpy as np
import pytest

from oracle import zipc_oracle as zo
import encoder_model as model
from zipc_b200 import _lib, synth
from zipc_b200 import zipc_deflate as zd

pytestmark = pytest.mark.gpu

HEAD = 256          # bytes in front of the first input of a buffer (the decoder's first refill starts 16-aligned before it)
TAIL = 4096 + 256   # bytes left unused after the last byte a test places or expects to be read
LEVELS = {"none": _lib.LEVEL_NONE, "fast": _lib.LEVEL_FAST, "default": _lib.LEVEL_DEFAULT, "best": _lib.LEVEL_BEST}
CK_ORACLE = {_lib.CK_NONE: zo.CRC_NOP, _lib.CK_ADLER32: zo.CRC_ADLER32, _lib.CK_CRC32: zo.CRC_CRC32}


@pytest.fixture(scope="module")
def ctx():
    c = zd.Context(0)
    zd.set_default_context(c)
    yield c
    zd.set_default_context(None)
    c.close()


# ---- device buffers through the library's own helpers ------------------------------------------------------------------
class DevBuf:
    """A device allocation (zipc_b200_dev_alloc) with a host image of what it must hold: a canary pattern everywhere, the
    placed items at their offsets.  upload() writes the image, read() returns the whole allocation."""

    def __init__(self, ctx, size, seed=0):
        self.ctx, self.size = ctx, size
        p = C.c_void_p()
        ctx._check(ctx.L.zipc_b200_dev_alloc(ctx.h, size, C.byref(p)), "dev_alloc")
        self.p = p.value
        self.image = np.random.default_rng(seed).integers(0, 256, size, dtype=np.uint8)
        self.canary = self.image.copy()

    def place(self, off, data):
        v = np.frombuffer(bytes(data), dtype=np.uint8)
        assert off >= 0 and off + v.size + TAIL <= self.size
        self.image[off:off + v.size] = v
        return off

    def upload(self, lo=0, hi=None):
        hi = self.size if hi is None else hi
        self.ctx._check(self.ctx.L.zipc_b200_memcpy_h2d(self.ctx.h, self.p + lo, self.image[lo:hi].ctypes.data, hi - lo), "memcpy_h2d")

    def read(self):
        out = np.empty(self.size, dtype=np.uint8)
        self.ctx._check(self.ctx.L.zipc_b200_memcpy_d2h(self.ctx.h, out.ctypes.data, self.p, self.size), "memcpy_d2h")
        return out

    def free(self):
        if self.p:
            self.ctx.L.zipc_b200_dev_free(self.ctx.h, self.p)
            self.p = None


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


def assert_untouched_outside(buf, got, ranges, what=""):
    """every byte of the allocation outside the given [lo, hi) ranges still holds the canary"""
    keep = np.ones(buf.size, dtype=bool)
    for lo, hi in ranges:
        keep[lo:hi] = False
    bad = np.flatnonzero((got != buf.canary) & keep)
    assert bad.size == 0, f"{what}: {bad.size} bytes changed outside the slots, first at {int(bad[0])}"


def source_layout(lengths, residues, start=HEAD):
    """offsets of inputs laid out one after the other (no gaps but for alignment), input i at residues[i] mod 16"""
    offs, pos = [], start
    for n, r in zip(lengths, residues):
        pos += (r - pos) % 16
        offs.append(pos)
        pos += n
    return offs, pos + TAIL


def slot_layout(caps, start, align=1, avoid16=False, odd=False):
    """output slots back to back from `start`; each offset rounded up to `align`, moved off multiples of 16 (avoid16) or
    onto odd addresses (odd), and an empty slot is followed by one byte -- the only gaps between slots"""
    offs, pos = [], start
    for cap in caps:
        pos += (-pos) % align
        if avoid16 and pos % 16 == 0:
            pos += align
        if odd and pos % 2 == 0:
            pos += 1
        offs.append(pos)
        pos += max(cap, 1)
    return offs, pos + TAIL


def _sz(vals):
    return (C.c_size_t * max(len(vals), 1))(*vals)


def deflate_dev(ctx, level, ck, mode, src, src_off, src_len, dst, dst_off, cap):
    n = len(src_off)
    dl, cs, st = (C.c_size_t * max(n, 1))(), (C.c_uint32 * max(n, 1))(), (C.c_int * max(n, 1))()
    rc = ctx.L.zipc_b200_deflate_batch_dev(ctx.h, LEVELS[level], ck, mode, n, src.p if src else None, _sz(src_off), _sz(src_len),
                                           dst.p if dst else None, _sz(dst_off), _sz(cap), dl, cs, st)
    return rc, list(dl[:n]), list(cs[:n]), list(st[:n])


def inflate_dev(ctx, ck, mode, src, src_off, src_len, dst, dst_off, max_out):
    n = len(src_off)
    dl, cs, st = (C.c_size_t * max(n, 1))(), (C.c_uint32 * max(n, 1))(), (C.c_int * max(n, 1))()
    rc = ctx.L.zipc_b200_inflate_batch_dev(ctx.h, ck, mode, n, src.p if src else None, _sz(src_off), _sz(src_len),
                                           dst.p if dst else None, _sz(dst_off), _sz(max_out), dl, cs, st)
    return rc, list(dl[:n]), list(cs[:n]), list(st[:n])


def oracle_inflate(s, cap, ck, mode):
    """(status, bytes, checksum) of the reference's inflate / inflate_and_crc_32 / inflate_and_adler_32"""
    try:
        out, c = zo.inflate_and_crc(bytes(s), cap, CK_ORACLE[ck])
    except zo.OracleError as e:
        return e.status, b"", 0
    if ck == _lib.CK_ADLER32 and mode == _lib.ADLER_RFC1950:
        c = zlib.adler32(out)
    return 0, out, c if ck != _lib.CK_NONE else 0


# ==== A. zipc_b200_deflate_batch_dev =====================================================================================
def _deflate_corpus():
    t = synth.text_v1(3, 140000).tobytes()
    rnd = synth.rand_v1(5, 70000).tobytes()
    items = [t[:n] for n in (0, 1, 3, 2047, 2048, 2049, 61439, 61440, 61441, 65536, 131077)]
    items += [synth.text_v1(1007, 300001).tobytes(), rnd, bytes(150000),
              b"".join(bytes([rnd[i]]) * (1 + rnd[i + 1] * 2) for i in range(0, 1200, 2)),
              synth.text_v1(11, (5 << 19) + 333).tobytes()]    # 2.5 MiB: one CTA encodes it (the dev path never splits)
    return items


_model_cache = {}


def model_deflate(data, level):
    key = (level, len(data), zlib.crc32(data))
    if key not in _model_cache:
        _model_cache[key] = zo.deflate(data, "none") if level == "none" else model.deflate(data, level)
    return _model_cache[key]


def _deflate_placed(ctx, dev, items, residues, level, ck=_lib.CK_CRC32, mode=_lib.ADLER_REF_COMPAT, caps=None):
    """items into one source buffer at the given residues, slots of deflate_bound (or caps) back to back at 4-aligned offsets
    that are no multiples of 16; -> (outputs, checksums, statuses, dst_len); checks the canary around the outputs"""
    offs, size = source_layout([len(d) for d in items], residues)
    src = dev(size, seed=1)
    for o, d in zip(offs, items):
        src.place(o, d)
    src.upload()
    caps = [ctx.L.zipc_b200_deflate_bound(len(d)) for d in items] if caps is None else caps
    doffs, dsize = slot_layout(caps, HEAD + 4, align=4, avoid16=True)
    dst = dev(dsize, seed=2)
    dst.upload()
    rc, dl, cs, st = deflate_dev(ctx, level, ck, mode, src, offs, [len(d) for d in items], dst, doffs, caps)
    assert rc == _lib.OK, (rc, ctx.L.zipc_b200_last_error(ctx.h))
    got = dst.read()
    ok = [i for i in range(len(items)) if st[i] == _lib.OK]
    assert_untouched_outside(dst, got, [(doffs[i], doffs[i] + (dl[i] if st[i] == _lib.OK else caps[i])) for i in range(len(items))], level)
    assert (src.read() == src.image).all(), "the input buffer changed"
    outs = [got[doffs[i]:doffs[i] + dl[i]].tobytes() if i in ok else None for i in range(len(items))]
    return outs, cs, st, dl


@pytest.mark.parametrize("level", ["none", "fast", "default", "best"])
def test_deflate_dev_equals_the_model_at_every_source_alignment(ctx, dev, level, monkeypatch):
    """every source residue mod 16 in one batch (bulk copies and plain loads side by side in the front end); every
    output equals the host encoder model's bytes (level None: the reference's stored blocks) and the host path's"""
    items = _deflate_corpus()
    first = [i % 16 for i in range(len(items))]
    for residues in (first, [7 if r == 0 else 0 for r in first]):   # (then the other way round: the aligned ones unaligned)
        outs, cs, st, _ = _deflate_placed(ctx, dev, items, residues, level)
        for i, d in enumerate(items):
            assert st[i] == _lib.OK and cs[i] == zlib.crc32(d), (i, residues[i])
            assert outs[i] == model_deflate(d, level), (i, len(d), residues[i])
    # the host entry point, every member on one CTA, gives the same bytes
    monkeypatch.setenv("ZIPC_B200_SPLIT_MIN", str(1 << 40))
    host = ctx.deflate_batch(items, level, _lib.CK_CRC32)
    for i, (hst, hout, hck) in enumerate(host):
        assert hst == _lib.OK and hout.tobytes() == outs[i] and hck == cs[i], i


@pytest.mark.parametrize("level", ["fast", "default", "best"])
def test_deflate_dev_prefix_views_see_no_continuation(ctx, dev, level):
    """members are views T[o:o+k] of one text in one buffer, so the bytes after each member are its own continuation"""
    t = synth.text_v1(41, 300000).tobytes()
    rng = np.random.default_rng(42)
    views = [(o, k) for o in (0, 1, 3, 4, 13, 16, 61440, 100003) for k in (1, 2, 3, 4, 5, 258, 259, 2049, 4093, 61439, 61441, 65537)]
    views += [(int(rng.integers(0, 150000)), int(rng.integers(1, 150000))) for _ in range(24)]
    src = dev(HEAD + len(t) + 64 + TAIL, seed=3)
    base = src.place(HEAD + 5, t)
    src.upload()
    caps = [ctx.L.zipc_b200_deflate_bound(k) for _, k in views]
    doffs, dsize = slot_layout(caps, HEAD + 8, align=4, avoid16=True)
    dst = dev(dsize, seed=4)
    dst.upload()
    rc, dl, cs, st = deflate_dev(ctx, level, _lib.CK_CRC32, 0, src, [base + o for o, _ in views], [k for _, k in views], dst, doffs, caps)
    assert rc == _lib.OK
    got = dst.read()
    for i, (o, k) in enumerate(views):
        d = t[o:o + k]
        assert st[i] == _lib.OK and cs[i] == zlib.crc32(d), (o, k)
        assert got[doffs[i]:doffs[i] + dl[i]].tobytes() == model_deflate(d, level), (o, k)
    assert_untouched_outside(dst, got, [(doffs[i], doffs[i] + dl[i]) for i in range(len(views))])


@pytest.mark.parametrize("level", ["fast", "default"])
def test_deflate_dev_stale_state_of_the_previous_member(ctx, dev, level):
    """600 prefixes of one 200 KB text at distinct lengths.  A CTA takes several members from the queue, longest first,
    so the ring and the hash chains it leaves behind hold the continuation of the member it encodes next."""
    t = synth.text_v1(43, 200000).tobytes()
    lens = sorted({int(x) for x in np.random.default_rng(44).integers(1, len(t) + 1, 640)})[:600]
    src = dev(HEAD + 2 * len(t) + 64 + TAIL, seed=5)
    a = src.place(HEAD, t)                       # one copy 16-aligned, one not: both staging branches
    b = src.place(HEAD + len(t) + 16 + 9, t)
    src.upload()
    caps = [ctx.L.zipc_b200_deflate_bound(n) for n in lens]
    doffs, dsize = slot_layout(caps, HEAD + 4, align=4, avoid16=True)
    dst = dev(dsize, seed=6)
    dst.upload()
    rc, dl, cs, st = deflate_dev(ctx, level, _lib.CK_NONE, 0, src, [a if i % 2 else b for i in range(len(lens))], lens, dst, doffs, caps)
    assert rc == _lib.OK
    got = dst.read()
    for i, n in enumerate(lens):
        assert st[i] == _lib.OK and cs[i] == 0, n
        assert got[doffs[i]:doffs[i] + dl[i]].tobytes() == model.deflate(t[:n], level), n


def _quirk_corpus():
    """as test_gpu_deflate._quirk_corpus: inputs on which the reference's Adler-32 differs from RFC 1950"""
    t = np.frombuffer(synth.text_v1(21, 300000).tobytes(), dtype=np.uint8)
    rnd = synth.rand_v1(22, 250001).tobytes()
    return [(t | 0x80).tobytes(), rnd, b"\xff" * 200000 + rnd[:5000] + b"\xff" * 70000,
            (t[:90000] | 0x80).tobytes() + rnd[:70000] + bytes(range(256)) * 300 + b"\xfe" * 65534 + t[:50000].tobytes(),
            bytes(range(256)) * 1000, b"\xff" * 5552, b""]


@pytest.mark.parametrize("level", ["none", "fast", "default", "best"])
def test_deflate_dev_checksums_of_the_input(ctx, dev, level):
    """CRC-32 = zlib; Adler-32 REF_COMPAT = the reference's fold over the output's blocks; RFC 1950 = zlib; CK_NONE = 0"""
    items = _quirk_corpus()
    residues = [3, 0, 9, 14, 1, 6, 11]
    outs, cs, st, _ = _deflate_placed(ctx, dev, items, residues, level, _lib.CK_CRC32)
    assert all(s == _lib.OK for s in st) and cs == [zlib.crc32(d) for d in items]
    outs, cs, st, _ = _deflate_placed(ctx, dev, items, residues, level, _lib.CK_ADLER32, _lib.ADLER_REF_COMPAT)
    quirk = 0
    for d, o, c, s in zip(items, outs, cs, st):
        back, ad = zo.inflate_and_adler_32(o)
        assert s == _lib.OK and back == d and c == ad
        quirk += c != zlib.adler32(d)
    assert quirk >= 3
    outs, cs, st, _ = _deflate_placed(ctx, dev, items, residues, level, _lib.CK_ADLER32, _lib.ADLER_RFC1950)
    assert all(s == _lib.OK for s in st) and cs == [zlib.adler32(d) for d in items]
    outs, cs, st, _ = _deflate_placed(ctx, dev, items, residues, level, _lib.CK_NONE)
    assert all(s == _lib.OK for s in st) and cs == [0] * len(items)


@pytest.mark.parametrize("level", ["none", "fast", "default", "best"])
def test_deflate_dev_bound_sized_slots_at_block_edges(ctx, dev, level):
    """random members of 61440 k +- 1 and 65534 k +- 1 bytes (stored blocks at every level) fit slots of
    zipc_b200_deflate_bound, as a caller sizes them"""
    sizes = [m * k + e for m in (61440, 65534) for k in (1, 2, 3, 5) for e in (-1, 1)]
    items = [synth.rand_v1(100 + i, n).tobytes() for i, n in enumerate(sizes)]
    outs, cs, st, _ = _deflate_placed(ctx, dev, items, [(5 * i) % 16 for i in range(len(items))], level)
    for d, o, s in zip(items, outs, st):
        assert s == _lib.OK and o == model_deflate(d, level), len(d)


@pytest.mark.parametrize("level", ["none", "default"])
def test_deflate_dev_slot_too_small(ctx, dev, level):
    """cap = exact gives the same bytes; exact - 1, - 3, - 4, - 5 and 0 give ZIPC_ERR_DST_TOO_SMALL with dst_len 0 and no
    write outside the slot, while the other members of the batch are still exact"""
    t = synth.text_v1(51, 400000).tobytes()
    rnd = synth.rand_v1(52, 70001).tobytes()
    items = [t[:n] for n in (1, 2, 3, 4, 5, 6, 7, 100, 2049, 61441, 131077)] + [t[7:300007], rnd, bytes(70000)]
    residues = [(3 * i) % 16 for i in range(len(items))]
    exact = [len(model_deflate(d, level)) for d in items]
    outs, cs, st, dl = _deflate_placed(ctx, dev, items, residues, level, caps=exact)
    assert st == [_lib.OK] * len(items) and dl == exact
    assert outs == [model_deflate(d, level) for d in items]
    for cut in (1, 3, 4, 5, None):
        # every third member gets the short slot (the buffer check of _deflate_placed covers the slot's neighbours)
        short = [i for i in range(len(items)) if (i + (cut or 0)) % 3 == 0]
        caps = [(0 if cut is None else max(0, exact[i] - cut)) if i in short else exact[i] for i in range(len(items))]
        outs, cs, st, dl = _deflate_placed(ctx, dev, items, residues, level, caps=caps)
        for i, d in enumerate(items):
            if i in short:
                assert st[i] == _lib.ERR_DST_TOO_SMALL and dl[i] == 0, (i, exact[i], caps[i])
            else:
                assert st[i] == _lib.OK and outs[i] == model_deflate(d, level) and cs[i] == zlib.crc32(d), i


def test_deflate_dev_arguments(ctx, dev):
    """a slot that is not 4-aligned is refused before anything runs; n = 0 is a no-op"""
    d = synth.text_v1(61, 10000).tobytes()
    src = dev(HEAD + len(d) + TAIL, seed=7)
    o = src.place(HEAD, d)
    src.upload()
    cap = ctx.L.zipc_b200_deflate_bound(len(d))
    dst = dev(HEAD + 2 * cap + TAIL, seed=8)
    dst.upload()
    for bad in (HEAD + 1, HEAD + 2, HEAD + 3):
        rc, _, _, _ = deflate_dev(ctx, "default", _lib.CK_CRC32, 0, src, [o, o], [len(d), len(d)], dst, [HEAD + cap + 4, bad], [cap, cap])
        assert rc == _lib.ERR_INVALID_ARG
    assert (dst.read() == dst.canary).all()
    assert deflate_dev(ctx, "default", _lib.CK_CRC32, 0, None, [], [], None, [], [])[0] == _lib.OK
    assert (dst.read() == dst.canary).all()


# ==== B. zipc_b200_inflate_batch_dev =====================================================================================
def _raw(data, level=6, strategy=zlib.Z_DEFAULT_STRATEGY, memlevel=8):
    c = zlib.compressobj(level, zlib.DEFLATED, -15, memlevel, strategy)
    return c.compress(data) + c.flush()


def _inflate_corpus(ctx):
    """(stream, decompressed size): zlib-made (all levels x strategies), oracle-made, made by this library, extreme code shapes"""
    rnd = np.random.default_rng(12)
    text = synth.text_v1(8, 120000).tobytes()
    r = synth.rand_v1(9, 40000).tobytes()
    datas = [text, r, bytes(60000), b"".join(bytes([r[i]]) * (1 + r[i + 1]) for i in range(0, 800, 2)),
             text[:30000] + r[:20000] + text[:30000], b"abc", b""]
    out = []
    for d in datas:
        for lvl in (0, 1, 6, 9):
            for strategy in (zlib.Z_DEFAULT_STRATEGY, zlib.Z_FIXED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE):
                out.append((_raw(d, lvl, strategy), d))
        for lvl in ("none", "fast", "default", "best"):
            out.append((zo.deflate(d, lvl), d))
    for level in ("fast", "default", "best"):
        for d, (st, cs, _) in zip(datas, ctx.deflate_batch(datas, level)):
            assert st == 0
            out.append((cs.tobytes(), d))
    # code shapes of test_gpu_inflate.test_extreme_code_shapes, smaller
    shapes = [np.minimum(rnd.exponential(s, 60000), 255).astype(np.uint8).tobytes() for s in (0.35, 1.4, 3.0)]
    shapes += [(b"\x00" * 1000 + b"\x01") * 60, bytes(rnd.integers(0, 2, 50000, dtype=np.uint8))]
    far = rnd.integers(0, 256, 33000, dtype=np.uint8).tobytes()
    shapes.append(far + far[:5000] + far[20000:29000] + far[:33000])
    for d in shapes:
        for lvl, strategy in ((9, zlib.Z_DEFAULT_STRATEGY), (1, zlib.Z_DEFAULT_STRATEGY), (6, zlib.Z_FILTERED), (6, zlib.Z_FIXED)):
            out.append((_raw(d, lvl, strategy), d))
        c = zlib.compressobj(6, zlib.DEFLATED, -15, 1)
        s = b"".join(c.compress(d[i:i + 1000]) + c.flush(zlib.Z_FULL_FLUSH if (i // 1000) % 2 else zlib.Z_SYNC_FLUSH)
                     for i in range(0, len(d), 1000)) + c.flush()
        out.append((s, d))
    return out


def _check_inflate_dev(ctx, dev, streams, caps, ck, mode, residues, odd=True, host=True):
    """one dev call; statuses, bytes and checksums against the oracle, the (status, dst_len, checksum) tuple against the host
    path, and no write outside [off, off + dst_len) (success) or [off, off + max_out) (failure).  -> statuses"""
    offs, size = source_layout([len(s) for s in streams], residues)
    src = dev(size, seed=11)
    for o, s in zip(offs, streams):
        src.place(o, s)
    src.upload()
    doffs, dsize = slot_layout(caps, HEAD + 1, odd=odd)
    dst = dev(dsize, seed=12)
    dst.upload()
    rc, dl, cs, st = inflate_dev(ctx, ck, mode, src, offs, [len(s) for s in streams], dst, doffs, caps)
    assert rc == _lib.OK, (rc, ctx.L.zipc_b200_last_error(ctx.h))
    got = dst.read()
    assert_untouched_outside(dst, got, [(doffs[i], doffs[i] + (dl[i] if st[i] == _lib.OK else caps[i])) for i in range(len(streams))],
                             f"ck {ck} mode {mode}")
    for i, s in enumerate(streams):
        est, eout, eck = oracle_inflate(s, caps[i], ck, mode)
        assert st[i] == est, (i, st[i], est, caps[i])
        if est == _lib.OK:
            assert dl[i] == len(eout) and got[doffs[i]:doffs[i] + dl[i]].tobytes() == eout, i
            assert cs[i] == eck, i
    if host:
        for i, (hst, hout, hck) in enumerate(ctx.inflate_batch(streams, caps, ck, mode)):
            assert (st[i], dl[i], cs[i]) == (hst, len(hout), hck), i
    return st


@pytest.mark.parametrize("ck,mode", [(_lib.CK_NONE, 0), (_lib.CK_CRC32, 0), (_lib.CK_ADLER32, _lib.ADLER_REF_COMPAT),
                                     (_lib.CK_ADLER32, _lib.ADLER_RFC1950)])
def test_inflate_dev_parity_with_the_oracle(ctx, dev, ck, mode):
    """every source residue mod 16, odd output offsets, slots back to back; max_out = exact, exact + 1, exact - 1 and 0,
    each stream through all four in turn"""
    corpus = _inflate_corpus(ctx)
    streams = [s for s, _ in corpus]
    for turn in range(4):
        caps = []
        for i, (_, d) in enumerate(corpus):
            v = (i + turn) % 4
            caps.append((len(d), len(d) + 1, max(0, len(d) - 1), 0)[v])
        st = _check_inflate_dev(ctx, dev, streams, caps, ck, mode, [(i + turn) % 16 for i in range(len(streams))])
        assert _lib.ERR_SIZE_EXCEEDED in st and _lib.OK in st


def _flushed_stream(data, every, level=6):
    """raw deflate of data with a Z_FULL_FLUSH after every `every` input bytes; -> (stream, byte offsets of the flush points)"""
    c = zlib.compressobj(level, zlib.DEFLATED, -15)
    out, marks = b"", []
    for i in range(0, len(data), every):
        out += c.compress(data[i:i + every])
        if i + every < len(data):
            out += c.flush(zlib.Z_FULL_FLUSH)
            marks.append(len(out))
    return out + c.flush(), marks


def _truncation_cases(ctx, dev, data, s, marks, par_min, spread=50):
    """members are views (start of S, len(S) - d) of one full stream S in the buffer: its continuation is in place"""
    L = len(s)
    cuts = sorted({L - d for d in range(1, 17)} | {L * k // (spread + 1) for k in range(1, spread + 1)} | {100, 1000, L // 2}
                  | {m + e for m in marks for e in (-1, 0, 1)})
    second = _raw(synth.text_v1(77, 5000).tobytes(), 6)
    buf_len = HEAD + L + len(second) + 64 + TAIL
    src = dev(buf_len, seed=21)
    a = src.place(HEAD + 3, s)
    src.place(a + L, second)            # S is followed by a second stream: trailing bytes, ignored by the reference
    src.upload()
    members = [(c, None) for c in cuts] + [(L, "full"), (L + len(second), "two")]
    for cap in (len(data), len(data) - 1):
        caps = [cap] * len(members)
        doffs, dsize = slot_layout(caps, HEAD + 1)
        dst = dev(dsize, seed=22)
        dst.upload()
        p0 = ctx.parallel_streams
        rc, dl, cs, st = inflate_dev(ctx, _lib.CK_CRC32, 0, src, [a] * len(members), [m for m, _ in members], dst, doffs, caps)
        p1 = ctx.parallel_streams
        assert rc == _lib.OK
        got = dst.read()
        want_par = 0
        for i, (n, kind) in enumerate(members):
            est, eout, eck = oracle_inflate(s[:n] if kind != "two" else s + second, cap, _lib.CK_CRC32, 0)
            assert st[i] == est, (n, L - n, cap, st[i], est)
            if kind is None:
                assert est == _lib.ERR_CORRUPTED if cap == len(data) else est != _lib.OK, (n, L - n, est)
            if est == _lib.OK:
                assert eout == data and got[doffs[i]:doffs[i] + dl[i]].tobytes() == data and cs[i] == zlib.crc32(data), n
                want_par += 1
        assert_untouched_outside(dst, got, [(doffs[i], doffs[i] + (dl[i] if st[i] == _lib.OK else caps[i])) for i in range(len(members))])
        if par_min == 0:
            assert p1 == p0, "the many-warp decoder ran"
        else:
            taken = sum(1 for n, _ in members if n >= par_min)
            assert p1[0] - p0[0] == want_par and p1[1] - p0[1] == taken - want_par, (p0, p1, taken, want_par)
            if cap == len(data):
                assert want_par == 2


def test_inflate_dev_truncated_views_one_warp(ctx, dev, monkeypatch):
    """One-warp decoder: a cut stream whose continuation follows it in memory is still "Corrupted data stream"
    (cuts d = 1..16 from the end, spread over the stream, and before / on / after full-flush block boundaries)"""
    monkeypatch.setenv("ZIPC_B200_PAR_MIN", "0")
    data = synth.text_v1(71, 400000).tobytes()
    s, marks = _flushed_stream(data, 50000)
    _truncation_cases(ctx, dev, data, s, marks, 0)
    # a stream that ends in a sync flush (no final block) and is cut there
    c = zlib.compressobj(6, zlib.DEFLATED, -15)
    body = c.compress(data[:100000]) + c.flush(zlib.Z_SYNC_FLUSH)
    whole = body + c.compress(data[100000:200000]) + c.flush()
    _truncation_cases(ctx, dev, data[:200000], whole, [len(body)], 0)


def test_inflate_dev_truncated_views_many_warps(ctx, dev, monkeypatch):
    """The same cuts on the many-warp decoder (block-start search, speculative chunks of 4 KiB): S is 1.4 MB compressed.
    Cut streams fall back to the one-warp decoder, which must give the same verdict."""
    monkeypatch.setenv("ZIPC_B200_PAR_MIN", "20000")
    monkeypatch.setenv("ZIPC_B200_PAR_CHUNK", "4096")
    data = synth.text_v1(72, 4 << 20).tobytes()
    s, marks = _flushed_stream(data, 1 << 20)
    assert len(s) >= 1 << 20
    _truncation_cases(ctx, dev, data, s, marks, 20000, spread=25)


def test_inflate_dev_large_streams_slot_bounds(ctx, dev, monkeypatch):
    """large streams on the many-warp decoder in slots back to back at odd offsets: max_out = exact decodes in parallel
    and writes its slot only; exact - 1 falls back to the one-warp decoder and reports SIZE_EXCEEDED"""
    monkeypatch.setenv("ZIPC_B200_PAR_MIN", "65536")
    datas = [synth.text_v1(81, 3 << 20).tobytes(), synth.text_v1(82, (2 << 20) + 777).tobytes()]
    streams = [_raw(d) for d in datas for _ in range(2)]
    caps = [len(datas[0]), len(datas[0]) - 1, len(datas[1]) - 1, len(datas[1])]
    p0 = ctx.parallel_streams
    st = _check_inflate_dev(ctx, dev, streams, caps, _lib.CK_CRC32, 0, [5, 0, 11, 2], host=False)
    p1 = ctx.parallel_streams
    assert st == [_lib.OK, _lib.ERR_SIZE_EXCEEDED, _lib.ERR_SIZE_EXCEEDED, _lib.OK]
    assert p1[0] - p0[0] == 2 and p1[1] - p0[1] == 2, (p0, p1)


def test_inflate_dev_same_pointer_new_bytes(ctx, dev):
    """stream A at pointer p with length L decodes through the many-warp decoder; the same range is overwritten with
    stream B (padded to L: trailing bytes are ignored) and decoded again with the same (p, L): the output is B's"""
    da = synth.text_v1(91, 2 << 20).tobytes()
    db = synth.text_v1(92, (2 << 20) - 4321).tobytes()
    sa, sb = _raw(da), _raw(db, 9)
    assert len(sb) < len(sa)
    L = len(sa)
    cap = len(da) + 1000                 # room for either output: a plan of A's would fit, so only the epoch protects B
    src = dev(HEAD + L + 64 + TAIL, seed=31)
    p = src.place(HEAD + 6, sa)
    src.upload()
    dst = dev(HEAD + cap + TAIL, seed=32)
    dst.upload()

    def decode(want):
        p0 = ctx.parallel_streams
        rc, dl, cs, st = inflate_dev(ctx, _lib.CK_CRC32, 0, src, [p], [L], dst, [HEAD + 3], [cap])
        assert rc == _lib.OK and st == [_lib.OK]
        assert ctx.parallel_streams[0] == p0[0] + 1, "not decoded by many warps"
        got = dst.read()
        assert dl[0] == len(want) and got[HEAD + 3:HEAD + 3 + dl[0]].tobytes() == want and cs[0] == zlib.crc32(want)

    for between in (False, True):
        src.place(p, sa)
        src.upload()
        decode(da)
        src.place(p, sb + bytes(L - len(sb)))
        src.upload(p, p + L)
        if between:
            assert zd.inflate(sa, decompressed_size=len(da)).get_ok() == da   # a host-path call in between
        decode(db)
    rc, _, _, _ = inflate_dev(ctx, _lib.CK_CRC32, 0, src, [p], [L], dst, [HEAD + 3], [_lib.SIZE_UNKNOWN])
    assert rc == _lib.ERR_INVALID_ARG


def test_inflate_dev_mixed_batch(ctx, dev):
    """dozens of small streams and two large ones in one call: all as the oracle says, the two large ones by many warps"""
    big = [synth.text_v1(61, 4 << 20).tobytes(), synth.text_v1(62, 3 << 20).tobytes()]
    small = [synth.text_v1(200 + i, 5000 + 777 * i).tobytes() for i in range(30)]
    datas = small[:12] + [big[0]] + small[12:] + [big[1]]
    streams = [_raw(d) if i % 3 else zo.deflate(d, "default") for i, d in enumerate(datas)]
    streams[12], streams[-1] = _raw(big[0]), _raw(big[1])
    p0 = ctx.parallel_streams
    _check_inflate_dev(ctx, dev, streams, [len(d) for d in datas], _lib.CK_CRC32, 0, [(7 * i) % 16 for i in range(len(datas))],
                       host=False)
    assert ctx.parallel_streams[0] == p0[0] + 2


# ==== C. checksum entry points ===========================================================================================
SIZES = [1, 2, 3, 4, 5, 15, 16, 17, 63, 64, 65, 127, 511, 512, 513, 1023, 4095, 4096, 4097, 5551, 5552, 5553,
         8191, 65535, 65536, 100003, 262144 + 7, 1 << 20, (1 << 20) + 13, 3 * 5552 * 16, 6 * 1024 * 1024 + 1]
EDGES = sorted({m * k + e for m in (4096, 5552) for k in (1, 2, 3, 7, 16, 33) for e in (-1, 1)})


def _crc_dev(ctx, p, n):
    out = C.c_uint32()
    ctx._check(ctx.L.zipc_b200_crc32_dev(ctx.h, p, n, C.byref(out)), "crc32_dev")
    return out.value


def _adler_dev(ctx, p, n, mode):
    out = C.c_uint32()
    ctx._check(ctx.L.zipc_b200_adler32_dev(ctx.h, p, n, mode, C.byref(out)), "adler32_dev")
    return out.value


def test_checksums_dev_sizes_and_all_alignments(ctx, dev):
    """crc32_dev, crc32_dev_async, adler32_dev (both flavours) at every source residue mod 16, on prefix views of a
    larger buffer (the bytes after each view are real data), at the sizes of test_gpu_checksums and around the CRC tile and
    the Adler chunk"""
    top = max(SIZES) + 16
    buf = dev(HEAD + top + TAIL, seed=41)
    data = synth.rand_v1(43, top)
    base = buf.place(HEAD, data.tobytes())
    buf.upload()
    word = dev(HEAD + 64 + TAIL, seed=42)
    word.upload()
    for n in SIZES + EDGES:
        for r in range(16):
            v = data[r:r + n]
            b = v.tobytes()
            crc = zlib.crc32(b)
            assert _crc_dev(ctx, buf.p + base + r, n) == crc, (n, r)
            ctx._check(ctx.L.zipc_b200_crc32_dev_async(ctx.h, buf.p + base + r, n, word.p + HEAD + 4), "crc32_dev_async")
            got = np.empty(4, dtype=np.uint8)
            ctx._check(ctx.L.zipc_b200_memcpy_d2h(ctx.h, got.ctypes.data, word.p + HEAD + 4, 4), "memcpy_d2h")
            assert int(got.view(np.uint32)[0]) == crc, (n, r)
            assert _adler_dev(ctx, buf.p + base + r, n, _lib.ADLER_RFC1950) == zlib.adler32(b), (n, r)
            assert _adler_dev(ctx, buf.p + base + r, n, _lib.ADLER_REF_COMPAT) == zo.adler32(b), (n, r)
    assert (buf.read() == buf.image).all()


def test_crc32_dev_async_writes_only_its_word(ctx, dev):
    """the async CRC lands in a caller's 4-byte word at a 4-aligned offset that is no multiple of 16, and nowhere else;
    two calls queued back to back are both right when read in stream order"""
    d = synth.text_v1(44, 300001).tobytes()
    src = dev(HEAD + len(d) + 64 + TAIL, seed=45)
    o = src.place(HEAD + 1, d)
    src.upload()
    out = dev(HEAD + 64 + TAIL, seed=46)
    out.upload()
    w1, w2 = HEAD + 4, HEAD + 40
    ctx._check(ctx.L.zipc_b200_crc32_dev_async(ctx.h, src.p + o, len(d), out.p + w1), "crc32_dev_async")
    ctx._check(ctx.L.zipc_b200_crc32_dev_async(ctx.h, src.p + o + 7, 5000, out.p + w2), "crc32_dev_async")
    got = out.read()
    assert int(got[w1:w1 + 4].view(np.uint32)[0]) == zlib.crc32(d)
    assert int(got[w2:w2 + 4].view(np.uint32)[0]) == zlib.crc32(d[7:5007])
    assert_untouched_outside(out, got, [(w1, w1 + 4), (w2, w2 + 4)])


def test_checksums_dev_of_nothing(ctx, dev):
    """a NULL source of length 0: CRC-32 0, Adler-32 1 (both flavours), and an async 0 written over a canary"""
    assert _crc_dev(ctx, None, 0) == 0
    assert _adler_dev(ctx, None, 0, _lib.ADLER_REF_COMPAT) == 1
    assert _adler_dev(ctx, None, 0, _lib.ADLER_RFC1950) == 1
    out = dev(HEAD + 64 + TAIL, seed=47)
    out.image[HEAD + 12:HEAD + 16] = 0xA5
    out.canary[HEAD + 12:HEAD + 16] = 0xA5
    out.upload()
    ctx._check(ctx.L.zipc_b200_crc32_dev_async(ctx.h, None, 0, out.p + HEAD + 12), "crc32_dev_async")
    got = out.read()
    assert got[HEAD + 12:HEAD + 16].tolist() == [0, 0, 0, 0]
    assert_untouched_outside(out, got, [(HEAD + 12, HEAD + 16)])
