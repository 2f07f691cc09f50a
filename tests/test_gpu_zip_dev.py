"""GPU parity of the device-resident archive entry points (zipc_b200_zip_parse_dev, zipc_b200_zip_extract_batch_dev) with
the host entry points (zipc_b200_zip_parse_ex, zipc_b200_zip_extract_batch), CPython's zipfile and zlib.

Archives are made here: torch.save, np.savez / np.savez_compressed, CPython zipfile (stored, deflated, force_zip64, data
descriptors, a full-length comment), the oracle and the reference's own fixture.  The buffers follow
test_gpu_device_entry_points: allocated with the library's helpers, canary-filled, read back whole; archives at every
residue mod 16, output slots back to back at odd offsets."""
import ctypes as C
import io
import random
import struct
import zipfile
import zlib

import numpy as np
import pytest

from oracle import zipc_oracle as zo
from test_gpu_device_entry_points import DevBuf, HEAD, TAIL, assert_untouched_outside, slot_layout, source_layout
from zipc_b200 import _lib, synth, zipc
from zipc_b200 import zipc_deflate as zd

pytestmark = pytest.mark.gpu

TILE = 256 << 10      # kStoredTile (common.cuh): the stored kernel cuts members into tiles of this many bytes
FLAGS = [zipc.ZIP_REFERENCE, zipc.ZIP_ALLOW_ZIP64]
ERR_ZIP_EOCD, ERR_ZIP_SHORT, ERR_ZIP_CDFH, ERR_ZIP_LFH = 22, 24, 26, 27     # (include/zipc_b200.h)
FIELDS = ("path_len", "is_dir", "mode", "mtime", "version_made_by", "version_needed", "gp_flags", "compression", "start",
          "compressed_size", "decompressed_size", "crc32")


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


# ---- the two parsers -----------------------------------------------------------------------------------------------------
class Parsed:
    """the member array of one parse (freed with close()) and its fields as comparable records: the path's bytes, FIELDS,
    and compressed_bytes relative to the archive's base (None: null)"""

    def __init__(self, L, st, p, n, base):
        self.L, self.st, self.p, self.n = L, st, p, n
        self.records = []
        for i in range(n):
            m = p[i]
            cb = None if not m.compressed_bytes else m.compressed_bytes - base
            self.records.append((C.string_at(m.path, m.path_len),) + tuple(getattr(m, f) for f in FIELDS) + (cb,))

    def close(self):
        if self.p:
            self.L.zipc_b200_free(C.cast(self.p, C.c_void_p))
            self.p = None


def parse_host(ctx, data, flags, keep):
    v = np.frombuffer(bytes(data), dtype=np.uint8)
    keep.append(v)
    p, n = C.POINTER(_lib.Member)(), C.c_size_t()
    base = v.ctypes.data if v.size else None
    st = ctx.L.zipc_b200_zip_parse_ex(base, v.size, flags, C.byref(p), C.byref(n))
    return Parsed(ctx.L, st, p if st == _lib.OK else None, n.value, base or 0)


def parse_dev(ctx, d_ptr, length, flags):
    p, n = C.POINTER(_lib.Member)(), C.c_size_t()
    st = ctx.L.zipc_b200_zip_parse_dev(ctx.h, d_ptr, length, flags, C.byref(p), C.byref(n))
    return Parsed(ctx.L, st, p if st == _lib.OK else None, n.value, d_ptr or 0)


def _cap(m):
    if m.is_dir or m.gp_flags & 1 or m.compression not in (0, 8):
        return 0
    return m.compressed_size if m.compression == 0 else m.decompressed_size


def extract_host(ctx, arr, n):
    """zipc_b200_zip_extract_batch -> [(status, bytes, found)]"""
    need = C.c_size_t()
    off, ln = (C.c_size_t * max(n, 1))(), (C.c_size_t * max(n, 1))()
    found, st = (C.c_uint32 * max(n, 1))(), (C.c_int * max(n, 1))()
    rc = ctx.L.zipc_b200_zip_extract_batch(ctx.h, arr, n, None, 0, C.byref(need), off, ln, found, st)
    assert rc in (_lib.OK, _lib.ERR_DST_TOO_SMALL), rc
    arena = np.empty(max(need.value, 1), dtype=np.uint8)
    if rc == _lib.ERR_DST_TOO_SMALL:
        ctx._check(ctx.L.zipc_b200_fetch(ctx.h, arena.ctypes.data, arena.size), "fetch")
    return [(st[i], arena[off[i]:off[i] + ln[i]].tobytes(), found[i]) for i in range(n)]


def extract_dev(ctx, dev, arr, n, seed=7):
    """zipc_b200_zip_extract_batch_dev into slots back to back at odd offsets; checks that nothing outside the slots that
    may be written changed -> [(status, bytes, found)], dst buffer, slot offsets"""
    caps = [_cap(arr[i]) for i in range(n)]
    doffs, dsize = slot_layout(caps, HEAD + 1, odd=True)
    dst = dev(dsize, seed=seed)
    dst.upload()
    dl, fo, st = (C.c_size_t * max(n, 1))(), (C.c_uint32 * max(n, 1))(), (C.c_int * max(n, 1))()
    rc = ctx.L.zipc_b200_zip_extract_batch_dev(ctx.h, arr, n, dst.p, _sz(doffs), dl, fo, st)
    assert rc == _lib.OK, (rc, ctx.L.zipc_b200_last_error(ctx.h))
    got = dst.read()
    ranges = []
    for i in range(n):
        if st[i] == _lib.OK:
            ranges.append((doffs[i], doffs[i] + dl[i]))
        elif caps[i]:      # a failure: writes stay inside the slot (a rejected member has no slot)
            ranges.append((doffs[i], doffs[i] + caps[i]))
        assert dl[i] <= caps[i], i
    assert_untouched_outside(dst, got, ranges, "extract_batch_dev")
    return [(st[i], got[doffs[i]:doffs[i] + dl[i]].tobytes(), fo[i]) for i in range(n)], dst, doffs


def check_archive(ctx, dev, data, flags, residues=(0,), zf_check=True, seed=3):
    """parse_dev == parse_ex field by field; extract_batch_dev == extract_batch == zipfile.read, at each residue"""
    keep = []
    hp = parse_host(ctx, data, flags, keep)
    assert hp.st == _lib.OK, hp.st
    host = extract_host(ctx, hp.p, hp.n)
    zf = zipfile.ZipFile(io.BytesIO(bytes(data))) if zf_check else None
    for r in residues:
        src = dev(HEAD + 16 + len(data) + TAIL, seed=seed + r)
        a = src.place(HEAD + r, data)
        src.upload()
        dp = parse_dev(ctx, src.p + a, len(data), flags)
        try:
            assert dp.st == _lib.OK and dp.records == hp.records, r
            got, _, _ = extract_dev(ctx, dev, dp.p, dp.n, seed=seed + 100 + r)
            assert got == host, r
            for rec, (st, out, found) in zip(dp.records, got):
                if rec[2]:
                    continue
                assert st == _lib.OK and found == zlib.crc32(out) == rec[-2], rec[0]
                if zf is not None:
                    assert out == zf.read(rec[0].decode()), rec[0]
            assert (src.read() == src.image).all(), "the archive changed"
        finally:
            dp.close()
    hp.close()
    return host


# ---- archives ------------------------------------------------------------------------------------------------------------
def _torch_archive():
    import torch
    g = torch.Generator().manual_seed(5)
    sd = {"w": torch.randn(300_000, generator=g), "b": torch.arange(1000, dtype=torch.int64),
          "u8": torch.randint(0, 255, (70_001,), generator=g, dtype=torch.uint8), "e": torch.empty(0),
          "h": torch.randn(3, 5, generator=g).half()}
    bio = io.BytesIO()
    torch.save(sd, bio)
    return bio.getvalue()


def _npz(compressed):
    rng = np.random.default_rng(6)
    arrays = {"a": rng.standard_normal(100_000), "b": np.arange(50_000, dtype=np.int32), "c": np.zeros(0),
              "t": np.frombuffer(synth.text_v1(7, 90_000).tobytes(), dtype=np.uint8)}
    bio = io.BytesIO()
    (np.savez_compressed if compressed else np.savez)(bio, **arrays)
    return bio.getvalue()


class _Unseekable(io.RawIOBase):   # makes zipfile write data descriptors (general purpose bit 3)
    def __init__(self):
        self.b = bytearray()

    def writable(self):
        return True

    def write(self, x):
        self.b += x
        return len(x)


def _cpython_archives():
    data = [synth.text_v1(50 + i, 20_000 + 7919 * i).tobytes() for i in range(4)] + [synth.rand_v1(60, 33_333).tobytes()]
    out = {}
    bio = io.BytesIO()
    with zipfile.ZipFile(bio, "w") as zf:
        for i, d in enumerate(data):
            zf.writestr("s/%d.bin" % i, d, compress_type=zipfile.ZIP_STORED if i % 2 else zipfile.ZIP_DEFLATED)
        zf.writestr("s/dir/", b"")
    out["mixed"] = bio.getvalue()
    bio = io.BytesIO()
    with zipfile.ZipFile(bio, "w", zipfile.ZIP_DEFLATED) as zf:
        for i, d in enumerate(data):
            with zf.open("z%d.txt" % i, "w", force_zip64=True) as fh:
                fh.write(d)
    out["force_zip64"] = bio.getvalue()
    u = _Unseekable()
    with zipfile.ZipFile(u, "w", zipfile.ZIP_DEFLATED) as zf:
        for i, d in enumerate(data):
            zf.writestr("g%d.txt" % i, d, compress_type=zipfile.ZIP_STORED if i % 2 else zipfile.ZIP_DEFLATED)
    out["descriptors"] = bytes(u.b)
    bio = io.BytesIO()
    with zipfile.ZipFile(bio, "w", zipfile.ZIP_STORED) as zf:   # the directory lies before the EOCD search window
        for i, d in enumerate(data):
            zf.writestr("c%d" % i, d[:3000])
        zf.comment = b"#" * 65535
    out["long_comment"] = bio.getvalue()
    return out


def _oracle_archive():
    ms = [zo.member_make(b"doc/a.txt", **zo.file_deflate_of_binary_string(synth.text_v1(70, 40_000).tobytes(), "default")),
          zo.member_make(b"doc/b.bin", **zo.file_stored_of_binary_string(synth.rand_v1(71, 5_000).tobytes())),
          zo.member_make(b"doc/", is_dir=True),
          zo.member_make(b"mimetype", **zo.file_stored_of_binary_string(b"application/x-test"))]
    return zo.zip_encode(ms)


# ==== real-world shapes ====================================================================================================
def test_torch_save_archive(ctx, dev):
    """a torch.save checkpoint: stored members, 64-byte aligned payloads, data descriptors; one tensor above the tile size"""
    data = _torch_archive()
    zf = zipfile.ZipFile(io.BytesIO(data))
    infos = zf.infolist()
    assert all(i.compress_type == zipfile.ZIP_STORED for i in infos) and all(i.flag_bits & 8 for i in infos if i.file_size)
    assert max(i.file_size for i in infos) > TILE
    for flags in FLAGS:
        check_archive(ctx, dev, data, flags, residues=range(16) if flags == zipc.ZIP_REFERENCE else (5,))


@pytest.mark.parametrize("compressed", [False, True])
def test_npz_archives(ctx, dev, compressed):
    data = _npz(compressed)
    methods = {i.compress_type for i in zipfile.ZipFile(io.BytesIO(data)).infolist()}
    assert methods == ({zipfile.ZIP_DEFLATED} if compressed else {zipfile.ZIP_STORED})
    for flags in FLAGS:
        check_archive(ctx, dev, data, flags, residues=range(16) if flags == zipc.ZIP_REFERENCE else (11,))


def test_reference_fixture_and_oracle_archive(ctx, dev, zip_docs):
    for flags in FLAGS:
        check_archive(ctx, dev, zip_docs, flags, residues=(0, 3, 14))
        check_archive(ctx, dev, _oracle_archive(), flags, residues=(1, 8))


@pytest.mark.parametrize("kind", ["mixed", "force_zip64", "descriptors", "long_comment"])
def test_cpython_archives(ctx, dev, kind):
    data = _cpython_archives()[kind]
    for flags in FLAGS:
        check_archive(ctx, dev, data, flags, residues=(2, 9, 15))


# ==== the stored kernel ====================================================================================================
def test_stored_member_edges_in_one_batch(ctx, dev):
    """stored members of 0, 1, 63, 64, 65 bytes and k * TILE - 1, k * TILE, k * TILE + 1, with deflate members and directories
    in the same archive and batch"""
    sizes = [0, 1, 15, 16, 17, 63, 64, 65, 511, 512, 513] + [k * TILE + d for k in (1, 2, 3) for d in (-1, 0, 1)]
    bio = io.BytesIO()
    datas = {}
    with zipfile.ZipFile(bio, "w") as zf:
        for i, n in enumerate(sizes):
            d = synth.rand_v1(80 + i, n).tobytes()
            datas["s%02d" % i] = d
            zf.writestr("s%02d" % i, d, compress_type=zipfile.ZIP_STORED)
            if i % 4 == 0:
                t = synth.text_v1(120 + i, 1000 + 5000 * i).tobytes()
                datas["t%02d" % i] = t
                zf.writestr("t%02d" % i, t, compress_type=zipfile.ZIP_DEFLATED)
                zf.writestr("d%02d/" % i, b"")
    data = bio.getvalue()
    host = check_archive(ctx, dev, data, zipc.ZIP_REFERENCE, residues=(0, 1, 7, 12))
    assert len(host) == len(datas) + len(sizes[::4]) and all(st == _lib.OK for st, _, _ in host)


def test_stored_phases_caller_built_members(ctx, dev):
    """caller-built stored members over one device buffer: every source residue against destination residues that run
    through all 16 phases, sizes below, at and above the warp path's 64 bytes and across a tile; found is zlib.crc32"""
    payloads = [synth.rand_v1(200 + i, n).tobytes() for i, n in
                enumerate([64, 65, 127, 128, 1000, 4097, 33_333, TILE + 77, 48, 3, 0, 100_003, 2 * TILE - 5, 600, 7777, 70])]
    n = len(payloads)
    for turn in range(2):
        src_res = [(i + turn) % 16 for i in range(n)]
        dst_res = [(5 * i + 3 + 9 * turn) % 16 for i in range(n)]
        offs, size = source_layout([len(p) for p in payloads], src_res)
        src = dev(size, seed=20 + turn)
        for o, p in zip(offs, payloads):
            src.place(o, p)
        src.upload()
        doffs, dsize = source_layout([len(p) for p in payloads], dst_res, start=HEAD + 1)
        dst = dev(dsize, seed=30 + turn)
        dst.upload()
        arr = (_lib.Member * n)()
        for i, p in enumerate(payloads):
            arr[i] = _lib.Member(None, 0, 0, 0o644, 315532800, 20, 20, 0, 0, src.p, offs[i], len(p), len(p), zlib.crc32(p), 0)
        dl, fo, st = (C.c_size_t * n)(), (C.c_uint32 * n)(), (C.c_int * n)()
        assert ctx.L.zipc_b200_zip_extract_batch_dev(ctx.h, arr, n, dst.p, _sz(doffs), dl, fo, st) == _lib.OK
        got = dst.read()
        assert_untouched_outside(dst, got, [(doffs[i], doffs[i] + len(p)) for i, p in enumerate(payloads)])
        for i, p in enumerate(payloads):
            assert (st[i], dl[i], fo[i]) == (_lib.OK, len(p), zlib.crc32(p)), (i, len(p), src_res[i], dst_res[i])
            assert got[doffs[i]:doffs[i] + len(p)].tobytes() == p, (i, len(p))


# ==== statuses =============================================================================================================
def _status_files():
    """the mix of test_gpu_zip.test_extract_statuses"""
    text = synth.text_v1(77, 50000).tobytes()
    cs = zo.deflate(text, "default")
    F = zipc.File.make
    files = [F(cs, compression=8, decompressed_size=len(text), decompressed_crc_32=zlib.crc32(text)).get_ok(),
             F(cs, compression=8, decompressed_size=len(text), decompressed_crc_32=1).get_ok(),
             F(cs, compression=8, decompressed_size=len(text) - 1, decompressed_crc_32=zlib.crc32(text)).get_ok(),
             F(cs[:100], compression=8, decompressed_size=len(text), decompressed_crc_32=5).get_ok(),
             F(cs, compression=8, decompressed_size=len(text), decompressed_crc_32=0, gp_flags=0x801).get_ok(),
             F(cs, compression=14, decompressed_size=len(text), decompressed_crc_32=0).get_ok(),
             zipc.File.stored_of_binary_string(text).get_ok(),
             F(text, compression=0, decompressed_size=len(text), decompressed_crc_32=5).get_ok()]
    want = [_lib.OK, _lib.ERR_CHECKSUM, _lib.ERR_SIZE_EXCEEDED, _lib.ERR_CORRUPTED, _lib.ERR_ZIP_ENCRYPTED, _lib.ERR_ZIP_FORMAT,
            _lib.OK, _lib.ERR_CHECKSUM]
    return text, files, want


def test_extract_statuses_archive(ctx, dev):
    """the status mix built into one archive, parsed on the device: every status, dst_len, found and byte as the host
    call's; the slots of the encrypted and the lzma member stay untouched"""
    text, files, want = _status_files()
    z = {}
    for i, f in enumerate(files):
        z = zipc.add(zipc.Member.make("m%d" % i, f).get_ok(), z)
    z = zipc.add(zipc.Member.make("dir/", None).get_ok(), z)
    data = zipc.to_binary_string(z).get_ok()
    keep = []
    hp = parse_host(ctx, data, zipc.ZIP_REFERENCE, keep)
    host = extract_host(ctx, hp.p, hp.n)
    src = dev(HEAD + 16 + len(data) + TAIL, seed=40)
    a = src.place(HEAD + 9, data)
    src.upload()
    dp = parse_dev(ctx, src.p + a, len(data), zipc.ZIP_REFERENCE)
    assert dp.st == _lib.OK and dp.records == hp.records
    got, _, _ = extract_dev(ctx, dev, dp.p, dp.n, seed=41)
    assert got == host
    assert [st for st, _, _ in got] == [_lib.OK] + want   # ("dir/" sorts first)
    assert got[1][1] == got[7][1] == text and got[8][1] == text and got[8][2] == zlib.crc32(text)
    dp.close()
    hp.close()


def test_extract_statuses_caller_built(ctx, dev):
    """the same mix as caller-built members over one device buffer, payloads at odd offsets"""
    text, files, want = _status_files()
    payloads = [bytes(f.compressed_bytes[f.start:f.start + f.compressed_size]) for f in files]
    offs, size = source_layout([len(p) for p in payloads], [3, 6, 9, 12, 15, 2, 5, 8])
    src = dev(size, seed=42)
    for o, p in zip(offs, payloads):
        src.place(o, p)
    src.upload()
    n = len(files)
    arr, harr = (_lib.Member * n)(), (_lib.Member * n)()
    views = [np.frombuffer(p, dtype=np.uint8) for p in payloads]
    for i, f in enumerate(files):
        common = (None, 0, 0, 0o644, 315532800, 20, 20, f.gp_flags, f.compression)
        tail = (len(payloads[i]), f.decompressed_size, f.decompressed_crc_32, 0)
        arr[i] = _lib.Member(*common, src.p, offs[i], *tail)
        harr[i] = _lib.Member(*common, views[i].ctypes.data, 0, *tail)
    host = extract_host(ctx, harr, n)
    got, _, _ = extract_dev(ctx, dev, arr, n, seed=43)
    assert got == host and [st for st, _, _ in got] == want
    assert got[0][1] == text and got[1][2] == zlib.crc32(text) and got[7][2] == zlib.crc32(text)


# ==== parser parity on corrupt archives ====================================================================================
def _small_archive(force):
    z = {}
    for i in range(5):
        d = synth.text_v1(90 + i, 3000 + 997 * i).tobytes()
        if i % 2:
            f = zipc.File.make(zlib.compress(d, 6)[2:-4], compression=8, decompressed_size=len(d), decompressed_crc_32=zlib.crc32(d)).get_ok()
        else:
            f = zipc.File.make(d, compression=0, decompressed_size=len(d), decompressed_crc_32=zlib.crc32(d)).get_ok()
        z = zipc.add(zipc.Member.make("dir/m%02d.txt" % i, f, mtime=1_700_000_000 + i).get_ok(), z)
    z = zipc.add(zipc.Member.make("dir/", None).get_ok(), z)
    return bytes(zipc.to_binary_string(z, zip64="force" if force else False).get_ok())


def _regions(s):
    """[lo, hi) of the EOCD, the central directory and every local header of a well-formed archive"""
    e = len(s) - 22
    cd = struct.unpack_from("<I", s, e + 16)[0]
    if cd == 0xFFFFFFFF:
        cd = struct.unpack_from("<Q", s, len(s) - 22 - 20 - 56 + 48)[0]
    out = [(e, len(s)), (cd, e)]
    o = 0
    while s[o:o + 4] == b"PK\x03\x04":   # (the writer's archives: sizes in the local headers, or in their ZIP64 extra field)
        out.append((o, o + 30))
        nlen, xlen = struct.unpack_from("<HH", s, o + 26)
        csize = struct.unpack_from("<I", s, o + 18)[0]
        if csize == 0xFFFFFFFF:
            csize = struct.unpack_from("<Q", s, o + 30 + nlen + 4 + 8)[0]
        o += 30 + nlen + xlen + csize
    return out


def _zip64_corruptions(s):
    """the corruptions of test_zip64_host.test_corrupt_zip64_records_are_refused"""
    out = []
    loc = len(s) - 22 - 20
    rec = loc - 56

    def put(fmt, at, *v):
        b = bytearray(s)
        struct.pack_into(fmt, b, at, *v)
        out.append(bytes(b))
    put("<Q", loc + 8, len(s) + 5)
    put("<I", loc + 16, 2)
    put("<QQ", rec + 24, 1 << 40, 1 << 40)
    put("<Q", rec + 48, len(s))
    cd = struct.unpack_from("<Q", s, rec + 48)[0]
    plen = struct.unpack_from("<H", s, cd + 28)[0]
    put("<H", cd + 46 + plen + 2, 8)
    put("<H", cd + 46 + plen, 0x7075)
    b = bytearray(s)
    b[-18] = b[-17] = 0xFF
    out.append(bytes(b))
    return out


def _mutants(s, rng, count):
    regions = _regions(s)
    out = []
    for _ in range(count):
        kind = rng.random()
        if kind < 0.15:
            out.append(s[:rng.randrange(0, len(s))])     # truncation
            continue
        lo, hi = regions[rng.randrange(len(regions))]
        at = rng.randrange(lo, hi)
        b = bytearray(s)
        b[at] = rng.choice([0, 0xFF, b[at] ^ (1 << rng.randrange(8)), (b[at] + 1) & 0xFF, (b[at] - 1) & 0xFF, rng.randrange(256)])
        out.append(bytes(b))
    return out


def test_parser_parity_on_corrupt_archives(ctx, dev):
    """a few hundred seeded single-byte changes of the EOCD, the directory and the local headers, truncations, and the ZIP64
    corruptions: parse_dev gives parse_ex's status every time, and the same members when it succeeds.  Bytes after a cut
    archive are the device buffer's canary, so a read past len would show."""
    rng = random.Random(1234)
    cases = []
    for force in (False, True):
        s = _small_archive(force)
        cases += [s] + _mutants(s, rng, 200)
        if force:
            cases += _zip64_corruptions(s)
    big = max(len(c) for c in cases)
    src = dev(HEAD + 16 + big + TAIL, seed=50)
    statuses = set()
    keep = []
    for k, c in enumerate(cases):
        src.image[:] = src.canary
        a = src.place(HEAD + k % 16, c)
        src.upload()
        for flags in FLAGS:
            hp = parse_host(ctx, c, flags, keep)
            dp = parse_dev(ctx, src.p + a, len(c), flags)
            assert dp.st == hp.st, (k, flags, dp.st, hp.st)
            if hp.st == _lib.OK:
                assert dp.records == hp.records, (k, flags)
            statuses.add(hp.st)
            hp.close()
            dp.close()
        keep.clear()
    assert {_lib.OK, ERR_ZIP_EOCD, ERR_ZIP_CDFH, ERR_ZIP_LFH} <= statuses and len(statuses) >= 6, statuses


# ==== fresh reads ==========================================================================================================
def test_rewritten_payload_is_read_again(ctx, dev):
    """a stored payload rewritten in device memory between two calls: the second reports ZIPC_ERR_CHECKSUM with found the
    CRC-32 of the new bytes, and its slot holds the new bytes"""
    old = synth.rand_v1(300, TILE + 1000).tobytes()
    bio = io.BytesIO()
    with zipfile.ZipFile(bio, "w") as zf:
        zf.writestr("p", old, compress_type=zipfile.ZIP_STORED)
    data = bio.getvalue()
    src = dev(HEAD + 16 + len(data) + TAIL, seed=60)
    a = src.place(HEAD + 4, data)
    src.upload()
    dp = parse_dev(ctx, src.p + a, len(data), zipc.ZIP_REFERENCE)
    assert dp.st == _lib.OK and dp.n == 1
    got, _, _ = extract_dev(ctx, dev, dp.p, 1, seed=61)
    assert got == [(_lib.OK, old, zlib.crc32(old))]
    start = a + dp.p[0].start
    new = bytearray(old)
    new[TILE + 3] ^= 0x40
    new = bytes(new)
    src.place(start, new)
    src.upload(start, start + len(new))
    got, _, _ = extract_dev(ctx, dev, dp.p, 1, seed=62)
    assert got == [(_lib.ERR_CHECKSUM, new, zlib.crc32(new))]
    dp.close()


# ==== arguments ============================================================================================================
def test_arguments(ctx, dev):
    data = _oracle_archive()
    src = dev(HEAD + 16 + len(data) + TAIL, seed=70)
    a = src.place(HEAD, data)
    src.upload()
    L, h = ctx.L, ctx.h
    p, n = C.POINTER(_lib.Member)(), C.c_size_t()
    # parse: NULL arguments, short archives, an archive that is only an EOCD
    assert L.zipc_b200_zip_parse_dev(None, src.p + a, len(data), 0, C.byref(p), C.byref(n)) == _lib.ERR_INVALID_ARG
    assert L.zipc_b200_zip_parse_dev(h, None, len(data), 0, C.byref(p), C.byref(n)) == _lib.ERR_INVALID_ARG
    assert L.zipc_b200_zip_parse_dev(h, src.p + a, len(data), 0, None, C.byref(n)) == _lib.ERR_INVALID_ARG
    assert L.zipc_b200_zip_parse_dev(h, src.p + a, len(data), 0, C.byref(p), None) == _lib.ERR_INVALID_ARG
    for k in (0, 1, 21):
        assert parse_dev(ctx, src.p + a, k, 0).st == ERR_ZIP_SHORT
    assert parse_dev(ctx, None, 0, 0).st == ERR_ZIP_SHORT
    only = b"PK\x05\x06" + bytes(18)
    e = src.place(HEAD + 4096 + 3, only)
    src.upload()
    keep = []
    for flags in FLAGS:
        dp, hp = parse_dev(ctx, src.p + e, len(only), flags), parse_host(ctx, only, flags, keep)
        assert dp.st == hp.st == _lib.OK and dp.n == hp.n == 0
        dp.close()
        hp.close()
    # extract: n = 0, NULL arrays, members whose payloads are host memory (pageable or pinned)
    dl, fo, st = (C.c_size_t * 8)(), (C.c_uint32 * 8)(), (C.c_int * 8)()
    dst = dev(HEAD + 200_000 + TAIL, seed=71)
    dst.upload()
    assert L.zipc_b200_zip_extract_batch_dev(h, None, 0, None, None, None, None, None) == _lib.OK
    dp = parse_dev(ctx, src.p + a, len(data), 0)
    assert dp.st == _lib.OK
    offs = _sz([HEAD + 1 + 50_000 * i for i in range(dp.n)])
    full = [h, dp.p, dp.n, dst.p, offs, dl, fo, st]
    for k in (0, 1, 3, 4, 5, 7):
        args = list(full)
        args[k] = None
        assert L.zipc_b200_zip_extract_batch_dev(*args) == _lib.ERR_INVALID_ARG, k
    assert L.zipc_b200_zip_extract_batch_dev(h, dp.p, dp.n, dst.p, offs, dl, None, st) == _lib.OK   # (found may be NULL)
    hp = parse_host(ctx, data, 0, keep)
    launches = ctx.launches
    dst.upload()
    assert L.zipc_b200_zip_extract_batch_dev(h, hp.p, hp.n, dst.p, offs, dl, fo, st) == _lib.ERR_INVALID_ARG
    pinned = C.c_void_p()
    assert L.zipc_b200_host_alloc(len(data), C.byref(pinned)) == _lib.OK
    C.memmove(pinned.value, data, len(data))
    mixed = (_lib.Member * dp.n)(*[dp.p[i] for i in range(dp.n)])
    for i in range(dp.n):
        if mixed[i].compressed_bytes:
            mixed[i].compressed_bytes = pinned.value
            break
    assert L.zipc_b200_zip_extract_batch_dev(h, mixed, dp.n, dst.p, offs, dl, fo, st) == _lib.ERR_INVALID_ARG
    L.zipc_b200_host_free(pinned)
    assert ctx.launches == launches, "something ran before the host pointer was refused"
    assert (dst.read() == dst.canary).all()
    hp.close()
    dp.close()
