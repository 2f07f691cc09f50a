"""GPU parity of the device-resident archive writer, zipc_b200_zip_deflate_archive_dev, with the host calls
(zipc_b200_zip_deflate_archive_ex, and zipc_b200_zip_assemble_ex over zipc_b200_deflate_batch for stored members),
CPython's zipfile, torch.load and the device-resident reader (zipc_b200_zip_parse_dev, zipc_b200_zip_extract_batch_dev).

The buffers follow test_gpu_device_entry_points: allocated with the library's helpers, canary-filled, read back whole.
Payloads sit at every residue mod 16, the archive at an odd offset of its buffer."""
import ctypes as C
import io
import struct
import zipfile
import zlib

import numpy as np
import pytest

from test_gpu_device_entry_points import DevBuf, HEAD, TAIL, assert_untouched_outside, source_layout
from zipc_b200 import _lib, synth
from zipc_b200 import zipc
from zipc_b200 import zipc_deflate as zd

pytestmark = pytest.mark.gpu

LEVELS = {"none": _lib.LEVEL_NONE, "fast": _lib.LEVEL_FAST, "default": _lib.LEVEL_DEFAULT, "best": _lib.LEVEL_BEST}
REF, ALLOW, FORCE = zipc.ZIP_REFERENCE, zipc.ZIP_ALLOW_ZIP64, zipc.ZIP_FORCE_ZIP64
ERR_ZIP_COUNT, ERR_ZIP_SIZE = 28, 30      # (include/zipc_b200.h)
STORED, DEFLATE = 0, 8


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


def _arr(typ, vals):
    return None if vals is None else (typ * max(len(vals), 1))(*vals)


class Paths:
    """host path arrays of one batch (paths, path_len)"""

    def __init__(self, paths):
        self.bufs = [C.create_string_buffer(p, max(len(p), 1)) for p in paths]
        self.pp = (C.c_void_p * max(len(paths), 1))(*[C.cast(b, C.c_void_p).value for b in self.bufs])
        self.pl = (C.c_uint32 * max(len(paths), 1))(*[len(p) for p in paths])


def bound(ctx, paths, lens, comp=None):
    return ctx.L.zipc_b200_zip_archive_bound(len(paths), Paths(paths).pl, _sz(lens), _arr(C.c_int32, comp))


def host_archive(ctx, level, paths, payloads, modes=None, mtimes=None, first=None, flags=REF):
    """zipc_b200_zip_deflate_archive_ex into pageable memory -> (rc, bytes)"""
    n = len(paths)
    p = Paths(paths)
    vs = [np.frombuffer(bytes(x), dtype=np.uint8) for x in payloads]
    sp = (C.c_void_p * max(n, 1))(*[v.ctypes.data if v.size else None for v in vs])
    cap = bound(ctx, paths, [v.size for v in vs])
    out = np.empty(cap, dtype=np.uint8)
    need = C.c_size_t()
    rc = ctx.L.zipc_b200_zip_deflate_archive_ex(ctx.h, LEVELS[level], n, p.pp, p.pl, sp, _sz([v.size for v in vs]),
                                                _arr(C.c_int32, modes), _arr(C.c_int64, mtimes), first, flags,
                                                out.ctypes.data, cap, C.byref(need))
    return rc, (out[:need.value].tobytes() if rc == _lib.OK else None)


def dev_archive(ctx, dev, level, paths, payloads, comp=None, modes=None, mtimes=None, first=None, flags=REF, cap=None,
                seed=0):
    """zipc_b200_zip_deflate_archive_dev with payload i at residue 3 i + 1 mod 16 and the archive at an odd offset; checks that
    the source is unchanged and that nothing outside the archive (everything, on failure) was written -> (rc, out_len,
    bytes)"""
    n = len(paths)
    lens = [len(x) for x in payloads]
    offs, size = source_layout(lens, [(3 * i + 1) % 16 for i in range(n)])
    src = dev(size, seed=seed)
    for o, x in zip(offs, payloads):
        src.place(o, x)
    src.upload()
    if cap is None:
        cap = bound(ctx, paths, lens, comp)
    at = HEAD + 1
    dst = dev(at + max(cap, 1) + TAIL, seed=seed + 1)
    dst.upload()
    p = Paths(paths)
    out_len = C.c_size_t()
    rc = ctx.L.zipc_b200_zip_deflate_archive_dev(ctx.h, LEVELS[level], n, p.pp, p.pl, src.p, _sz(offs), _sz(lens),
                                                 _arr(C.c_int32, comp), _arr(C.c_int32, modes), _arr(C.c_int64, mtimes),
                                                 first, flags, dst.p + at, cap, C.byref(out_len))
    got = dst.read()
    assert (src.read() == src.image).all(), "the payloads changed"
    if rc != _lib.OK:
        assert (got == dst.canary).all(), f"rc {rc}: the output buffer was written"
        return rc, out_len.value, None
    assert out_len.value <= cap
    assert_untouched_outside(dst, got, [(at, at + out_len.value)], "zip_deflate_archive_dev")
    return rc, out_len.value, got[at:at + out_len.value].tobytes()


def same(got, want):
    """byte for byte, or where the first difference is"""
    if got != want:
        k = next((i for i, (a, b) in enumerate(zip(got, want)) if a != b), min(len(got), len(want)))
        raise AssertionError(f"{len(got)} bytes against {len(want)}, first difference at {k}: "
                             f"{got[max(k - 8, 0):k + 24].hex()} against {want[max(k - 8, 0):k + 24].hex()}")


# ---- members -------------------------------------------------------------------------------------------------------------
def _text(seed, n):
    return synth.text_v1(seed, n).tobytes()


def _rand(seed, n):
    return synth.rand_v1(seed, n).tobytes()


def _batch():
    """16 members (every source residue): duplicate paths, "mimetype" in the middle, backslash paths, empty payloads, sizes
    around one block (61,440) and one stored block / 64 KiB"""
    items = [(b"b/second.txt", _text(1, 5_000)), (b"dup", _text(2, 300)), (b"a\\win\\path.txt", _text(3, 61_439)),
             (b"empty", b""), (b"z/61440", _text(4, 61_440)), (b"mimetype", b"application/x-test"),
             (b"custom/first", _text(5, 1_234)), (b"z/61441", _rand(6, 61_441)), (b"z/65535", _text(7, 65_535)),
             (b"dup", _rand(8, 999)), (b"z/65536", _text(9, 65_536)), (b"z/65537", _rand(10, 65_537)),
             (b"", b"no name"), (b"a/empty2", b""), (b"c\\d", _text(11, 20_000)), (b"y", _rand(12, 777))]
    paths = [p for p, _ in items]
    payloads = [d for _, d in items]
    modes = [0o644, 0o600, 0o755, 0o7777, 0o640, 0o444, 0o644, 0o600, 0o755, 0o711, 0o644, 0o600, 0o700, 0o644, 0o755, 0o640]
    mtimes = [1_700_000_000, 0, 100_000_000, 315_532_799, 315_532_800, 4_000_000_000, 1_234_567_890, -5, 946_684_800,
              1_600_000_001, 1_500_000_000, 1_000_000_000, 2_000_000_000, 1_111_111_111, 1_222_222_222, 1_333_333_333]
    return paths, payloads, modes, mtimes


# ==== 1. all members deflated: the host call's bytes ======================================================================
@pytest.mark.parametrize("level", list(LEVELS))
@pytest.mark.parametrize("flags", [REF, ALLOW, FORCE])
def test_equal_to_the_host_call(ctx, dev, level, flags):
    paths, payloads, modes, mtimes = _batch()
    k = list(LEVELS).index(level) + flags
    first = None if k % 2 else b"custom/first"
    if k % 3 == 0:
        modes = mtimes = None
    rc, want = host_archive(ctx, level, paths, payloads, modes, mtimes, first, flags)
    assert rc == _lib.OK
    for comp in (None, [DEFLATE] * len(paths)):
        rc, n, got = dev_archive(ctx, dev, level, paths, payloads, comp, modes, mtimes, first, flags, seed=k)
        assert rc == _lib.OK
        same(got, want)
    zf = zipfile.ZipFile(io.BytesIO(got))
    assert zf.testzip() is None
    names = [i.filename for i in zf.infolist()]
    assert names[0] == (first or b"mimetype").decode() and "a/win/path.txt" in names and names.count("dup") == 1
    assert zf.read("dup") == payloads[9]


# ==== 2. stored and deflated members in one archive =======================================================================
def _assemble(members, first, flags):
    arr, _keep = zipc._to_c(members)
    cap = 1 << 24
    out = np.empty(cap, dtype=np.uint8)
    n = C.c_size_t()
    rc = _lib.lib().zipc_b200_zip_assemble_ex(arr, len(members), first, flags, out.ctypes.data, cap, C.byref(n))
    assert rc == _lib.OK
    return out[:n.value].tobytes()


@pytest.mark.parametrize("level", ["none", "default"])
@pytest.mark.parametrize("flags", [REF, FORCE])
def test_mixed_stored_and_deflated(ctx, dev, level, flags):
    paths, payloads, modes, mtimes = _batch()
    paths = [p.replace(b"\\", b"/") for p in paths]
    comp = [STORED if i % 3 != 1 else DEFLATE for i in range(len(paths))]
    comp[paths.index(b"z/65537")] = STORED
    defl = [i for i in range(len(paths)) if comp[i] == DEFLATE]
    res = ctx.deflate_batch([payloads[i] for i in defl], level, _lib.CK_CRC32)
    files = {}
    for i, (st, cs, crc) in zip(defl, res):
        assert st == _lib.OK
        files[i] = zipc.File.make(bytes(cs), compression=DEFLATE, decompressed_size=len(payloads[i]), decompressed_crc_32=crc).get_ok()
    for i in range(len(paths)):
        if comp[i] == STORED:
            files[i] = zipc.File.make(payloads[i], compression=STORED, decompressed_size=len(payloads[i]),
                                      decompressed_crc_32=zlib.crc32(payloads[i])).get_ok()
    members = [zipc.Member.make(paths[i], files[i], modes[i], mtimes[i]).get_ok() for i in range(len(paths))]
    want = _assemble(members, None, flags)
    rc, n, got = dev_archive(ctx, dev, level, paths, payloads, comp, modes, mtimes, None, flags, seed=20 + flags)
    assert rc == _lib.OK
    same(got, want)
    zf = zipfile.ZipFile(io.BytesIO(got))
    assert zf.testzip() is None
    last = {p: d for p, d in zip(paths, payloads)}
    for info in zf.infolist():
        assert zf.read(info) == last[info.filename.encode()]
        i = max(k for k in range(len(paths)) if paths[k] == info.filename.encode())
        assert info.compress_type == (zipfile.ZIP_STORED if comp[i] == STORED else zipfile.ZIP_DEFLATED)
    # the device-resident reader gives the payloads back
    a = dev(HEAD + 16 + len(got) + TAIL, seed=30)
    at = a.place(HEAD + 7, got)
    a.upload()
    p, cnt = C.POINTER(_lib.Member)(), C.c_size_t()
    assert ctx.L.zipc_b200_zip_parse_dev(ctx.h, a.p + at, len(got), ALLOW, C.byref(p), C.byref(cnt)) == _lib.OK
    caps = [p[i].compressed_size if p[i].compression == STORED else p[i].decompressed_size for i in range(cnt.value)]
    offs, size = source_layout(caps, [5] * cnt.value)
    d = dev(size, seed=31)
    d.upload()
    dl, fo, st = (C.c_size_t * cnt.value)(), (C.c_uint32 * cnt.value)(), (C.c_int * cnt.value)()
    assert ctx.L.zipc_b200_zip_extract_batch_dev(ctx.h, p, cnt.value, d.p, _sz(offs), dl, fo, st) == _lib.OK
    out = d.read()
    for i in range(cnt.value):
        data = last[C.string_at(p[i].path, p[i].path_len)]
        assert st[i] == _lib.OK and out[offs[i]:offs[i] + dl[i]].tobytes() == data and fo[i] == zlib.crc32(data)
    ctx.L.zipc_b200_free(C.cast(p, C.c_void_p))


# ==== 3. a torch.save checkpoint written in device memory ================================================================
def test_checkpoint_round_trip(ctx, dev):
    import torch
    g = torch.Generator().manual_seed(3)
    sd = {"w": torch.randn(200_000, generator=g), "i": torch.arange(5000, dtype=torch.int64),
          "u8": torch.randint(0, 255, (300_001,), generator=g, dtype=torch.uint8), "h": torch.randn(7, 9, generator=g).half(),
          "e": torch.empty(0)}
    bio = io.BytesIO()
    torch.save(sd, bio)
    zf = zipfile.ZipFile(io.BytesIO(bio.getvalue()))
    paths = [i.filename.encode() for i in zf.infolist()]
    payloads = [zf.read(i) for i in zf.infolist()]
    for comp in ([STORED] * len(paths), [DEFLATE] * len(paths)):
        rc, n, got = dev_archive(ctx, dev, "default", paths, payloads, comp, seed=40 + comp[0])
        assert rc == _lib.OK
        back = torch.load(io.BytesIO(got))
        assert back.keys() == sd.keys()
        for k in sd:
            assert back[k].dtype == sd[k].dtype and torch.equal(back[k], sd[k]), k


# ==== 4. large members cut into primed segments ===========================================================================
def test_split_members(ctx, dev, monkeypatch):
    paths = [b"big3m", b"mid400k", b"small"]
    payloads = [_text(50, 3 << 20), _text(51, 400 << 10), _text(52, 10_000)]
    rc, want = host_archive(ctx, "default", paths, payloads)
    assert rc == _lib.OK
    rc, n, got = dev_archive(ctx, dev, "default", paths, payloads, seed=50)
    assert rc == _lib.OK and got == want
    monkeypatch.setenv("ZIPC_B200_SPLIT_MIN", str(1 << 40))   # the same members on one CTA each: other streams
    try:
        rc, n, whole = dev_archive(ctx, dev, "default", paths, payloads, seed=52)
        assert rc == _lib.OK and whole != want
        assert whole == host_archive(ctx, "default", paths, payloads)[1]
    finally:
        monkeypatch.delenv("ZIPC_B200_SPLIT_MIN")
    for a in (got, whole):
        zf = zipfile.ZipFile(io.BytesIO(a))
        assert [zf.read(p.decode()) for p in paths] == payloads


# ==== 5. bound and capacity ===============================================================================================
@pytest.mark.parametrize("level", ["none", "default"])
def test_bound_and_capacity(ctx, dev, level):
    paths = [b"r", b"big/incompressible", b"t", b"\\x"]
    payloads = [_rand(60, 100), _rand(61, 2 << 20), _text(62, 3000), b""]
    for comp in (None, [DEFLATE, DEFLATE, STORED, STORED]):
        b = bound(ctx, paths, [len(x) for x in payloads], comp)
        rc, need, got = dev_archive(ctx, dev, level, paths, payloads, comp, flags=FORCE, seed=60)
        assert rc == _lib.OK and need <= b
        rc, n2, exact = dev_archive(ctx, dev, level, paths, payloads, comp, flags=FORCE, cap=need, seed=62)
        assert rc == _lib.OK and n2 == need and exact == got
        rc, n3, none = dev_archive(ctx, dev, level, paths, payloads, comp, flags=FORCE, cap=need - 1, seed=64)
        assert rc == _lib.ERR_DST_TOO_SMALL and n3 == need and none is None
    assert bound(ctx, [], [], None) == 56 + 20 + 22


# ==== 6. ZIP64 ============================================================================================================
def test_zip64_member_count(ctx, dev):
    n = 66_000
    paths = [b"m/%06d" % (i * 7919 % n) for i in range(n)]
    payloads = [bytes([i & 0xFF]) * (i % 13) for i in range(n)]
    rc, want = host_archive(ctx, "fast", paths, payloads, flags=ALLOW)
    assert rc == _lib.OK
    rc, _, got = dev_archive(ctx, dev, "fast", paths, payloads, flags=ALLOW, seed=70)
    assert rc == _lib.OK and got == want
    comp = [STORED if i % 2 else DEFLATE for i in range(n)]
    for c in (None, comp):
        rc, _, got = dev_archive(ctx, dev, "fast", paths, payloads, c, flags=REF, seed=72)
        assert rc == ERR_ZIP_COUNT and got is None


def test_zip64_stored_member_of_4_gib(ctx):
    import torch
    big = (4 << 30) + 17
    n_src = big + 64
    torch.cuda.manual_seed(9)
    src = torch.empty(n_src, dtype=torch.uint8, device="cuda:0").random_(0, 256)
    at = 3
    paths = [b"a", b"huge.bin", b"z"]
    offs, lens = [0, at, at + big], [1, big, 40]
    comp = [DEFLATE, STORED, STORED]
    cap = bound(ctx, paths, lens, comp)
    out = torch.full((cap + 64,), 0x5A, dtype=torch.uint8, device="cuda:0")
    p = Paths(paths)
    out_len = C.c_size_t()
    L, h = ctx.L, ctx.h

    def write(flags, pos):
        return L.zipc_b200_zip_deflate_archive_dev(h, _lib.LEVEL_DEFAULT, 3, p.pp, p.pl, src.data_ptr(), _sz(offs), _sz(lens),
                                                   _arr(C.c_int32, comp), None, None, None, flags, out.data_ptr() + pos, cap,
                                                   C.byref(out_len))
    assert write(REF, 1) == ERR_ZIP_SIZE
    torch.cuda.synchronize()
    assert bool((out == 0x5A).all())
    assert write(ALLOW, 1) == _lib.OK
    total = out_len.value
    arch = out[1:1 + total]
    assert bool((out[1 + total:] == 0x5A).all()) and int(out[0]) == 0x5A
    # the device-resident reader: the member comes back whole, its CRC-32 that of another kernel over the source
    mp, cnt = C.POINTER(_lib.Member)(), C.c_size_t()
    assert L.zipc_b200_zip_parse_dev(h, arch.data_ptr(), total, ALLOW, C.byref(mp), C.byref(cnt)) == _lib.OK and cnt.value == 3
    assert [C.string_at(mp[i].path, mp[i].path_len) for i in range(3)] == [b"a", b"huge.bin", b"z"]
    m = mp[1]
    assert m.compression == STORED and m.compressed_size == m.decompressed_size == big
    want_crc = C.c_uint32()
    assert L.zipc_b200_crc32_dev(h, src.data_ptr() + at, big, C.byref(want_crc)) == _lib.OK
    assert m.crc32 == want_crc.value
    dst = torch.empty(big + 1, dtype=torch.uint8, device="cuda:0")
    dl, fo, st = (C.c_size_t * 1)(), (C.c_uint32 * 1)(), (C.c_int * 1)()
    one = (_lib.Member * 1)(m)
    assert L.zipc_b200_zip_extract_batch_dev(h, one, 1, dst.data_ptr(), _sz([1]), dl, fo, st) == _lib.OK
    assert st[0] == _lib.OK and dl[0] == big and fo[0] == want_crc.value
    assert bool(torch.equal(dst[1:], src[at:at + big]))
    # the host parser over the headers and directory, downloaded around the payload
    data_end = m.start + big
    head, tail = arch[:m.start].cpu().numpy(), arch[data_end:].cpu().numpy()
    host = np.zeros(total, dtype=np.uint8)
    host[:m.start], host[data_end:] = head, tail
    L.zipc_b200_free(C.cast(mp, C.c_void_p))
    hp, hn = C.POINTER(_lib.Member)(), C.c_size_t()
    assert L.zipc_b200_zip_parse_ex(host.ctypes.data, total, ALLOW, C.byref(hp), C.byref(hn)) == _lib.OK and hn.value == 3
    assert (hp[1].compressed_size, hp[1].decompressed_size, hp[1].crc32, hp[1].start) == (big, big, want_crc.value, m.start)
    assert (hp[2].start, hp[2].compressed_size) == (data_end + 31, 40)
    L.zipc_b200_free(C.cast(hp, C.c_void_p))
    # the fields themselves: the local header's ZIP64 extra holds both sizes
    head, tail = head.tobytes(), tail.tobytes()
    lfh = m.start - (30 + 8 + 20)
    assert head[lfh:lfh + 4] == b"PK\x03\x04" and head[lfh + 30:lfh + 38] == b"huge.bin"
    assert struct.unpack_from("<II", head, lfh + 18) == (0xFFFFFFFF, 0xFFFFFFFF)
    assert struct.unpack_from("<HHQQ", head, lfh + 38) == (1, 16, big, big)
    # the end records: EOCD with 32-bit fields saturated, locator, ZIP64 end record with the directory
    assert tail[-22:-18] == b"PK\x05\x06" and tail[-42:-38] == b"PK\x06\x07" and tail[-98:-94] == b"PK\x06\x06"
    count, cd_size, cd_start = struct.unpack_from("<QQQ", tail, len(tail) - 98 + 32)
    assert struct.unpack_from("<HHII", tail, len(tail) - 22 + 8) == (3, 3, cd_size, 0xFFFFFFFF)
    assert count == 3 and cd_start + cd_size == total - 98 and struct.unpack_from("<Q", tail, len(tail) - 42 + 8)[0] == cd_start + cd_size
    cd = cd_start - data_end
    # directory entries: "a" plain (47 bytes), "huge.bin" with both sizes in its extra, "z" with its local header offset
    assert tail[cd:cd + 4] == b"PK\x01\x02" and tail[cd + 46:cd + 47] == b"a"
    e = cd + 47
    assert struct.unpack_from("<II", tail, e + 20) == (0xFFFFFFFF, 0xFFFFFFFF) and tail[e + 46:e + 54] == b"huge.bin"
    assert struct.unpack_from("<HHQQ", tail, e + 54) == (1, 16, big, big)
    z = e + 46 + 8 + 20
    assert struct.unpack_from("<I", tail, z + 42)[0] == 0xFFFFFFFF and tail[z + 46:z + 47] == b"z"
    assert struct.unpack_from("<HHQ", tail, z + 47) == (1, 8, data_end)
    assert z + 47 + 12 == cd + cd_size
    del src, out, arch, dst
    torch.cuda.empty_cache()


# ==== 7. arguments ========================================================================================================
def test_arguments(ctx, dev):
    L, h = ctx.L, ctx.h
    paths, payloads = [b"x", b"y"], [_text(80, 1000), b"abc"]
    offs, size = source_layout([1000, 3], [1, 2])
    src = dev(size, seed=80)
    for o, x in zip(offs, payloads):
        src.place(o, x)
    src.upload()
    cap = bound(ctx, paths, [1000, 3])
    dst = dev(HEAD + cap + TAIL, seed=81)
    dst.upload()
    p = Paths(paths)
    out_len = C.c_size_t()
    full = [h, _lib.LEVEL_DEFAULT, 2, p.pp, p.pl, src.p, _sz(offs), _sz([1000, 3]), None, None, None, None, REF,
            dst.p + HEAD + 1, cap, C.byref(out_len)]
    launches = ctx.launches
    for k in (0, 3, 4, 5, 6, 7, 13, 15):
        args = list(full)
        args[k] = None
        assert L.zipc_b200_zip_deflate_archive_dev(*args) == _lib.ERR_INVALID_ARG, k
    for level in (-1, 4):
        args = list(full)
        args[1] = level
        assert L.zipc_b200_zip_deflate_archive_dev(*args) == _lib.ERR_INVALID_ARG, level
    for bad in (1, 9, -1, 12):
        args = list(full)
        args[8] = _arr(C.c_int32, [STORED, bad])
        assert L.zipc_b200_zip_deflate_archive_dev(*args) == _lib.ERR_INVALID_ARG, bad
    hsrc = np.frombuffer(src.image.tobytes(), dtype=np.uint8)
    args = list(full)
    args[5] = hsrc.ctypes.data
    assert L.zipc_b200_zip_deflate_archive_dev(*args) == _lib.ERR_INVALID_ARG
    hout = np.zeros(cap, dtype=np.uint8)
    args = list(full)
    args[13] = hout.ctypes.data
    assert L.zipc_b200_zip_deflate_archive_dev(*args) == _lib.ERR_INVALID_ARG
    assert not hout.any()
    assert ctx.launches == launches, "something ran before the arguments were refused"
    assert (dst.read() == dst.canary).all()
    assert L.zipc_b200_zip_deflate_archive_dev(*full) == _lib.OK
    # n = 0: the host call's empty archive (22 bytes, 98 with ZIP64 records forced)
    for flags in (REF, FORCE):
        rc, want = host_archive(ctx, "default", [], [], flags=flags)
        assert rc == _lib.OK and len(want) == (22 if flags == REF else 98)
        e = dev(HEAD + 200 + TAIL, seed=82 + flags)
        e.upload()
        n0 = C.c_size_t()
        assert L.zipc_b200_zip_deflate_archive_dev(h, _lib.LEVEL_DEFAULT, 0, None, None, None, None, None, None, None, None,
                                                   None, flags, e.p + HEAD + 3, 200, C.byref(n0)) == _lib.OK
        got = e.read()
        assert n0.value == len(want) and got[HEAD + 3:HEAD + 3 + n0.value].tobytes() == want
        assert_untouched_outside(e, got, [(HEAD + 3, HEAD + 3 + n0.value)], "empty archive")
