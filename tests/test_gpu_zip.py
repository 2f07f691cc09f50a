"""GPU parity for the archive paths: Zipc.of_binary_string + File.to_binary_string (C3) and
File.deflate_of_binary_string + Zipc.to_binary_string (C4), through the `zipc` mirror module."""
import io
import zipfile
import zlib

import numpy as np
import pytest

from oracle import zipc_oracle as zo
from zipc_b200 import _lib, synth, zipc
from zipc_b200 import zipc_deflate as zd

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ctx():
    c = zd.Context(0)
    zd.set_default_context(c)
    yield c
    zd.set_default_context(None)
    c.close()


def _assert_zip(archive, original):  # test/test.ml:74-108
    z = zipc.of_binary_string(archive).get_ok()
    d = zipc.find("zip-docs/", z)
    assert d.kind is None and zo.ptime_to_date_time(d.mtime) == ((2023, 10, 21), (15, 6, 50)) and d.mode == 0o755
    r = zipc.find("zip-docs/rfc1951.txt", z)
    a = zipc.find("zip-docs/APPNOTE.TXT", z)
    assert zo.ptime_to_date_time(r.mtime) == ((2023, 10, 21), (15, 6, 24)) and r.mode == 0o644
    assert zo.ptime_to_date_time(a.mtime) == ((2023, 10, 21), (15, 6, 50)) and a.mode == 0o644
    if original:
        assert r.kind.compression == zipc.DEFLATE and r.kind.decompressed_size == 36944
        assert a.kind.compression == zipc.DEFLATE and a.kind.decompressed_size == 174585
    assert r.kind.decompressed_crc_32 == 0xFB4F3400 and a.kind.decompressed_crc_32 == 0x39B029C4
    rs, as_ = zipc.File.to_binary_strings([r.kind, a.kind])
    return z, rs.get_ok(), as_.get_ok()


def test_crunched_trip(ctx, zip_docs):  # test/test.ml:57-118, every codec step on the GPU
    z, r, a = _assert_zip(zip_docs, True)
    ms = {m.path: m for m in zo.zip_decode(zip_docs)}
    assert r == zo.file_to_binary_string(ms[b"zip-docs/rfc1951.txt"]) and a == zo.file_to_binary_string(ms[b"zip-docs/APPNOTE.TXT"])
    # redeflate_recode (test.ml:58-73)
    out = zipc.empty()
    files = [m for m in z.values() if m.kind is not None and zipc.File.can_extract(m.kind)]
    datas = [x.get_ok() for x in zipc.File.to_binary_strings([m.kind for m in files])]
    news = zipc.File.deflate_of_binary_strings(datas, level="best")
    for m in z.values():
        if m.kind is None:
            out = zipc.add(m, out)
    for m, f in zip(files, news):
        out = zipc.add(zipc.Member.make(m.path, f.get_ok(), mode=m.mode, mtime=m.mtime).get_ok(), out)
    recoded = zipc.to_binary_string(out).get_ok()
    assert len(recoded) == zipc.encoding_size(out)
    _z2, r2, a2 = _assert_zip(recoded, True)
    assert (r2, a2) == (r, a)
    # the oracle (reference decoder) and Info-ZIP-compatible zipfile read it too
    back = {m.path: m for m in zo.zip_decode(recoded)}
    assert zo.file_to_binary_string(back[b"zip-docs/APPNOTE.TXT"]) == a
    assert zipfile.ZipFile(io.BytesIO(recoded)).testzip() is None


def test_archive_layout_bit_exact_given_same_payloads(ctx):
    """X-2..X-4: with identical payloads the archive bytes equal the oracle's to_binary_string."""
    datas = [synth.text_v1(50 + i, 3000 + 777 * i).tobytes() for i in range(12)]
    files = [f.get_ok() for f in zipc.File.deflate_of_binary_strings(datas, level="default")]
    z = zipc.empty()
    oms = []
    for i, (d, f) in enumerate(zip(datas, files)):
        path = ("m/%05d.txt" % i) if i != 5 else "mimetype"
        z = zipc.add(zipc.Member.make(path, f, mtime=1697900810 + i).get_ok(), z)
        oms.append(zo.member_make(path.encode(), mtime=1697900810 + i, compression=8, compressed_bytes=bytes(f.compressed_bytes),
                                  decompressed_size=len(d), crc32=f.decompressed_crc_32))
    z = zipc.add(zipc.Member.make("dir\\sub", None).get_ok(), z)
    oms.append(zo.member_make(b"dir\\sub", is_dir=True))
    s = zipc.File.stored_of_binary_string(b"stored payload").get_ok()
    z = zipc.add(zipc.Member.make("s.bin", s, mode=0o600).get_ok(), z)
    oms.append(zo.member_make(b"s.bin", mode=0o600, **zo.file_stored_of_binary_string(b"stored payload")))
    for first in (None, "s.bin"):
        ours = zipc.to_binary_string(z, first=first).get_ok()
        assert ours == zo.zip_encode(oms, first.encode() if first else None)
    zf = zipfile.ZipFile(io.BytesIO(zipc.to_binary_string(z).get_ok()))
    assert zf.testzip() is None and zf.read("m/00003.txt") == datas[3]


def test_extract_statuses(ctx):
    text = synth.text_v1(77, 50000).tobytes()
    cs = zo.deflate(text, "default")
    good = zipc.File.make(cs, compression=8, decompressed_size=len(text), decompressed_crc_32=zlib.crc32(text)).get_ok()
    badcrc = zipc.File.make(cs, compression=8, decompressed_size=len(text), decompressed_crc_32=1).get_ok()
    small = zipc.File.make(cs, compression=8, decompressed_size=len(text) - 1, decompressed_crc_32=zlib.crc32(text)).get_ok()
    corrupt = zipc.File.make(cs[:100], compression=8, decompressed_size=len(text), decompressed_crc_32=0).get_ok()
    enc = zipc.File.make(cs, compression=8, decompressed_size=len(text), decompressed_crc_32=0, gp_flags=0x801).get_ok()
    lzma = zipc.File.make(cs, compression=14, decompressed_size=len(text), decompressed_crc_32=0).get_ok()
    stored = zipc.File.stored_of_binary_string(text).get_ok()
    storedbad = zipc.File.make(text, compression=0, decompressed_size=len(text), decompressed_crc_32=5).get_ok()
    res = zipc.File.to_binary_strings([good, badcrc, small, corrupt, enc, lzma, stored, storedbad])
    assert res[0].get_ok() == text and res[6].get_ok() == text
    assert res[1].message == "Checksum mismatch, expected 1 found %x)" % zlib.crc32(text)
    assert res[2].message == "deflate: Expected decompression size exceeded"
    assert res[3].message == "deflate: Corrupted data stream"
    assert res[4].message == "Encrypted file not supported"
    assert res[5].message == "Compression lzma not supported"
    assert res[7].message == "Checksum mismatch, expected 5 found %x)" % zlib.crc32(text)
    # same verdicts from the oracle
    for f, r in zip([good, badcrc, small, corrupt, stored, storedbad], [res[0], res[1], res[2], res[3], res[6], res[7]]):
        m = zo.member_make(b"x", compression=f.compression, compressed_bytes=bytes(f.compressed_bytes),
                           decompressed_size=f.decompressed_size, crc32=f.decompressed_crc_32)
        try:
            zo.file_to_binary_string(m); ok = True
        except zo.OracleError as e:
            ok = False
            assert e.message == r.message
        assert ok == r.is_ok()
    assert zipc.File.to_binary_string_no_crc_check(badcrc).get_ok() == (text, zlib.crc32(text))


def test_archive_of_binary_strings_c4_small(ctx):
    """C4 scaled down: 300 members compressed on the GPU and assembled; framing bit-exact vs the oracle's
    framing of the same payloads, every member inflates through the oracle, zipfile reads the archive."""
    sizes = synth.member_sizes(300, seed=4)
    datas = [synth.text_v1(3000 + i, int(n)).tobytes() for i, n in enumerate(sizes)]
    paths = ["m/%05d.txt" % i for i in range(300)]
    for level in ("fast", "default"):
        arch = zipc.archive_of_binary_strings(paths, datas, level=level).get_ok()
        ms = zo.zip_decode(arch)
        assert [m.path.decode() for m in ms] == paths
        assert zo.zip_encode(ms) == arch  # layout rules: re-encoding the decoded members reproduces the bytes
        for m, d in list(zip(ms, datas))[::17]:
            assert zo.file_to_binary_string(m) == d
        zf = zipfile.ZipFile(io.BytesIO(arch))
        assert zf.testzip() is None
        # and back through our own archive decode + batch extract
        z = zipc.of_binary_string(arch).get_ok()
        outs = zipc.File.to_binary_strings([z[p.encode()].kind for p in paths])
        assert all(o.get_ok() == d for o, d in zip(outs, datas))


def test_of_binary_string_errors(ctx, zip_docs):
    assert zipc.of_binary_string(b"").message == "File too short to be a ZIP archive"
    assert zipc.of_binary_string(bytes(100)).message == "Likely not a ZIP archive: no end of central directory record found"
    assert zipc.string_has_magic(zip_docs) and not zipc.string_has_magic(b"nope")


def test_box_wide_entry_points(ctx):
    """zipc_b200_mctx: every visible GPU behind one call (1 on the default test box; the same test runs under
    gpurun --gpus N).  Results are in input order and bit-exact with the single-device path and the oracle."""
    import zlib
    from zipc_b200 import synth
    m = zd.MultiContext(0)
    try:
        assert m.devices >= 1
        sizes = synth.member_sizes(120, seed=4)
        datas = [synth.text_v1(500 + i, int(n)) if i % 7 else synth.rand_v1(500 + i, int(n)) for i, n in enumerate(sizes)]
        datas += [np.zeros(0, dtype=np.uint8), synth.text_v1(1, 3)]
        res = m.deflate_batch(datas, "default", _lib.CK_CRC32)
        for d, (st, cs, crc) in zip(datas, res):
            assert st == 0 and crc == zlib.crc32(d.tobytes()) and zo.inflate(cs.tobytes()) == d.tobytes()
        back = m.inflate_batch([r[1] for r in res], [d.size for d in datas], _lib.CK_CRC32)
        for d, r, (st, out, crc) in zip(datas, res, back):
            assert st == 0 and crc == r[2] and out.tobytes() == d.tobytes()
        # per-member status survives the partitioning
        bad = [r[1].copy() for r in res[:8]]
        bad[3][len(bad[3]) // 2] ^= 0x55
        got = m.inflate_batch(bad, [d.size for d in datas[:8]], _lib.CK_CRC32)
        one = ctx.inflate_batch(bad, [d.size for d in datas[:8]], _lib.CK_CRC32)  # parity-tested against the oracle elsewhere
        assert [(a[0], a[2], a[1].tobytes()) for a in got] == [(b[0], b[2], b[1].tobytes()) for b in one]
        big = synth.rand_v1(77, (64 << 20) + 12345)
        assert m.crc32(big) == zlib.crc32(big.tobytes()) == zo.crc32(big.tobytes())
        assert m.crc32(b"") == 0 and m.crc32(b"a") == zlib.crc32(b"a")
        assert m.launches > 0
    finally:
        m.close()


def test_large_batches_are_pipelined_and_equal(ctx):
    """A large host-pointer batch WITH a caller arena runs in groups on sub-contexts (copies under the kernels): same
    results, same order, arena offsets consistent.  1,600 members, 100 MB."""
    import ctypes as C
    import zlib
    from zipc_b200 import synth
    L = ctx.L
    n = 1600
    datas = [synth.text_v1(7000 + i, 40_000 + (i * 7919) % 50_000) for i in range(n)]
    U = sum(d.size for d in datas)
    assert U > (64 << 20)
    src = np.concatenate(datas)
    offs = np.concatenate([[0], np.cumsum([d.size for d in datas])[:-1]]).astype(np.uint64)
    slen = np.array([d.size for d in datas], dtype=np.uint64)
    ptrs = (C.c_void_p * n)(*[src.ctypes.data + int(o) for o in offs])
    P = lambda a, t: a.ctypes.data_as(C.POINTER(t))
    arena = np.zeros(U // 2 + 16 * n + 4096, dtype=np.uint8)
    need = C.c_size_t(); off = np.zeros(n, dtype=np.uint64); dl = np.zeros(n, dtype=np.uint64)
    ck = np.zeros(n, dtype=np.uint32); st = np.zeros(n, dtype=np.int32)
    l0 = ctx.launches
    rc = L.zipc_b200_deflate_batch(ctx.h, 2, 2, 0, n, ptrs, P(slen, C.c_size_t), arena.ctypes.data, arena.size, C.byref(need),
                                   P(off, C.c_size_t), P(dl, C.c_size_t), P(ck, C.c_uint32), P(st, C.c_int))
    assert rc == 0 and (st == 0).all() and ctx.launches > l0
    assert need.value <= arena.size and int(off[-1] + dl[-1]) <= need.value
    assert (np.diff(off.astype(np.int64)) > 0).all()      # input order kept
    streams = []
    for i in (0, 1, n // 3, n // 2, n - 2, n - 1):
        cs = arena[int(off[i]):int(off[i]) + int(dl[i])].tobytes()
        assert zlib.decompress(cs, -15) == datas[i].tobytes() and int(ck[i]) == zlib.crc32(datas[i])
    # and back: inflate all members from the arena into a second arena
    cptrs = (C.c_void_p * n)(*[arena.ctypes.data + int(o) for o in off])
    out = np.zeros(U + 16 * n + 4096, dtype=np.uint8)
    ooff = np.zeros(n, dtype=np.uint64); ol = np.zeros(n, dtype=np.uint64); ck2 = np.zeros(n, dtype=np.uint32)
    rc = L.zipc_b200_inflate_batch(ctx.h, 2, 0, n, cptrs, P(dl, C.c_size_t), P(slen, C.c_size_t), out.ctypes.data, out.size, C.byref(need),
                                   P(ooff, C.c_size_t), P(ol, C.c_size_t), P(ck2, C.c_uint32), P(st, C.c_int))
    assert rc == 0 and (st == 0).all() and (ol == slen).all() and (ck2 == ck).all()
    for i in range(0, n, 97):
        assert out[int(ooff[i]):int(ooff[i]) + int(ol[i])].tobytes() == datas[i].tobytes()


def test_inflate_progressive_download_and_split_upload(ctx):
    """A large inflate batch from pinned memory into a pinned arena: the upload goes in two halves, the streams are decoded in
    download order (by output size, the late half's behind the others) and every group's arena range is copied out while the
    kernel still runs.  Offsets are the library's choice: they must tile the arena without overlap; contents, lengths,
    checksums and the statuses of damaged members must be those of the plain path."""
    import ctypes as C
    import zlib
    from zipc_b200 import synth
    L = ctx.L
    n = 2400
    datas = [synth.text_v1(9000 + i, 20_000 + (i * 7919) % 90_000).tobytes() for i in range(n)]
    U = sum(len(d) for d in datas)
    assert U > (128 << 20)
    comp = []
    for i, d in enumerate(datas):
        co = zlib.compressobj(6, zlib.DEFLATED, -15)
        comp.append(co.compress(d) + co.flush())
    bad = {5: "flip", n // 2 + 3: "flip", n - 7: "cut"}
    for i, how in bad.items():
        c = bytearray(comp[i])
        if how == "flip":
            c[len(c) // 2] ^= 0x5A
            c[len(c) // 2 + 1] ^= 0xC3
        else:
            c = c[: len(c) // 2]
        comp[i] = bytes(c)
    Ctot = sum(len(c) for c in comp)
    assert Ctot > (40 << 20)
    hsrc = C.c_void_p(); hdst = C.c_void_p()
    cap = U + 16 * n + 4096
    assert L.zipc_b200_host_alloc(Ctot + 64, C.byref(hsrc)) == 0 and L.zipc_b200_host_alloc(cap, C.byref(hdst)) == 0
    try:
        src = np.ctypeslib.as_array(C.cast(hsrc, C.POINTER(C.c_uint8)), shape=(Ctot + 64,))
        dst = np.ctypeslib.as_array(C.cast(hdst, C.POINTER(C.c_uint8)), shape=(cap,))
        dst[:] = 0xEE
        offs = np.zeros(n, dtype=np.uint64); t = 0
        for i, c in enumerate(comp):
            offs[i] = t; src[t:t + len(c)] = np.frombuffer(c, dtype=np.uint8); t += len(c)
        clen = np.array([len(c) for c in comp], dtype=np.uint64)
        ulen = np.array([len(d) for d in datas], dtype=np.uint64)
        ptrs = (C.c_void_p * n)(*[hsrc.value + int(o) for o in offs])
        P = lambda a, ty: a.ctypes.data_as(C.POINTER(ty))
        need = C.c_size_t(); ooff = np.zeros(n, dtype=np.uint64); ol = np.zeros(n, dtype=np.uint64)
        ck = np.zeros(n, dtype=np.uint32); st = np.zeros(n, dtype=np.int32)
        for rep in range(2):  # twice: the serial numbers and flags of the first call must not leak into the second
            rc = L.zipc_b200_inflate_batch(ctx.h, 2, 0, n, ptrs, P(clen, C.c_size_t), P(ulen, C.c_size_t), hdst, cap, C.byref(need),
                                           P(ooff, C.c_size_t), P(ol, C.c_size_t), P(ck, C.c_uint32), P(st, C.c_int))
            assert rc == 0 and need.value <= cap
            # the slots tile the arena: sorted by offset, each starts where the previous one's 16-byte aligned slot ends
            order = np.argsort(ooff, kind="stable")
            ends = ooff[order] + ((ulen[order] + 15) & ~np.uint64(15))
            assert int(ooff[order][0]) == 0 and (ooff[order][1:] == ends[:-1]).all() and int(ends[-1]) == need.value
            assert not (np.diff(ooff.astype(np.int64)) > 0).all()   # (download order, not input order: the progressive path ran)
            for i in range(n):
                if i in bad:  # (a flipped byte may still be a valid stream: then the checksum tells)
                    assert (st[i] != 0 and ol[i] == 0) or int(ck[i]) != zlib.crc32(datas[i]), (i, st[i])
                    continue
                assert st[i] == 0 and ol[i] == ulen[i]
                if i % 41 == 0 or i < 4 or i > n - 4:
                    assert dst[int(ooff[i]):int(ooff[i]) + int(ol[i])].tobytes() == datas[i]
                assert int(ck[i]) == zlib.crc32(datas[i])
            dst[:] = 0x11
    finally:
        L.zipc_b200_host_free(hsrc); L.zipc_b200_host_free(hdst)


def test_zip_extract_progressive_download_with_mixed_members(ctx):
    """zipc_b200_zip_extract_batch of a large archive into a pinned arena: the deflate members are decoded in download order
    and copied out group by group while the kernel runs, with stored members, directories and a deflate member whose
    directory CRC-32 is wrong between them.  The arena holds the deflate members by ascending output size, then the others
    in member order; every member's bytes, status and found are those of zipfile / zlib, and a second call on the same
    context gives the same results."""
    import ctypes as C
    L = ctx.L
    n = 1200
    buf = io.BytesIO()
    with zipfile.ZipFile(buf, "w", zipfile.ZIP_DEFLATED) as zw:   # (paths in member order: the parser returns members by path)
        for i in range(n):
            if i % 97 == 40:
                zw.mkdir("%04d-d" % i)
            elif i % 13 == 6:
                zw.writestr("%04d-s.bin" % i, synth.rand_v1(20_000 + i, 1 + (i * 7919) % 70_000).tobytes(), compress_type=zipfile.ZIP_STORED)
            else:
                zw.writestr("%04d-m.txt" % i, synth.text_v1(20_000 + i, 40_000 + (i * 6151) % 60_000).tobytes())
    arch = np.frombuffer(buf.getvalue(), dtype=np.uint8)
    zf = zipfile.ZipFile(io.BytesIO(buf.getvalue()))
    p, cnt = C.POINTER(_lib.Member)(), C.c_size_t()
    assert L.zipc_b200_zip_parse_ex(arch.ctypes.data, arch.size, zipc.ZIP_REFERENCE, C.byref(p), C.byref(cnt)) == _lib.OK
    hdst = C.c_void_p()
    try:
        assert cnt.value == n
        names = [C.string_at(p[i].path, p[i].path_len).decode() for i in range(n)]
        assert all(name.startswith("%04d-" % i) for i, name in enumerate(names))
        kind = ["dir" if p[i].is_dir else "stored" if p[i].compression == 0 else "deflate" for i in range(n)]
        want = [b"" if k == "dir" else zf.read(name) for k, name in zip(kind, names)]
        deflated = [i for i in range(n) if kind[i] == "deflate"]
        bad = deflated[len(deflated) // 2]
        p[bad].crc32 ^= 0x1
        # the arena the progressive download lays out: deflate members by (output size, index), then the rest in member order
        exp_off, t = np.zeros(n, dtype=np.uint64), 0
        for i in sorted(deflated, key=lambda i: (len(want[i]), i)) + [i for i in range(n) if kind[i] != "deflate"]:
            exp_off[i] = t
            t += (len(want[i]) + 15) & ~15
        assert len(deflated) >= 1024 and t >= (64 << 20) and {"dir", "stored"} <= set(kind)
        cap = t + 4096
        assert L.zipc_b200_host_alloc(cap, C.byref(hdst)) == 0
        dst = np.ctypeslib.as_array(C.cast(hdst, C.POINTER(C.c_uint8)), shape=(cap,))
        P = lambda a, ty: a.ctypes.data_as(C.POINTER(ty))
        runs = []
        for fill in (0xEE, 0x11):
            dst[:] = fill
            need = C.c_size_t()
            off, ln = np.zeros(n, dtype=np.uint64), np.zeros(n, dtype=np.uint64)
            fo, st = np.zeros(n, dtype=np.uint32), np.zeros(n, dtype=np.int32)
            rc = L.zipc_b200_zip_extract_batch(ctx.h, p, n, hdst, cap, C.byref(need), P(off, C.c_size_t), P(ln, C.c_size_t),
                                               P(fo, C.c_uint32), P(st, C.c_int))
            assert rc == _lib.OK and need.value == t
            assert (off == exp_off).all() and not (np.diff(off[deflated].astype(np.int64)) > 0).all()
            for i in range(n):
                assert st[i] == (_lib.ERR_CHECKSUM if i == bad else _lib.OK), (i, kind[i], st[i])
                assert ln[i] == len(want[i]) and fo[i] == (zlib.crc32(want[i]) if kind[i] != "dir" else 0), (i, kind[i])
                assert dst[int(off[i]):int(off[i]) + int(ln[i])].tobytes() == want[i], (i, kind[i])
            runs.append((off, ln, fo, st))
        assert all((a == b).all() for a, b in zip(*runs))
    finally:
        L.zipc_b200_free(C.cast(p, C.c_void_p))
        if hdst.value:
            L.zipc_b200_host_free(hdst)


def test_large_archive_pipelined_equals_plain(ctx):
    """zipc_b200_zip_deflate_archive of a large member set given in path order goes through the pipeline (every group's
    payloads copied to their archive offsets while later groups are compressed); given in reverse order it takes the plain
    path.  Zipc.to_binary_string writes members in path order either way: the two archives are the same bytes."""
    import io
    import zipfile
    from zipc_b200 import synth, zipc
    from zipc_b200 import zipc_deflate as zd
    zd.set_default_context(ctx)
    n = 1500
    datas = [synth.text_v1(5000 + i, 30_000 + (i * 6151) % 60_000) for i in range(n)]
    assert sum(d.size for d in datas) > (64 << 20)
    paths = ["big/%05d.txt" % i for i in range(n)]
    l0 = ctx.launches
    a = zipc.archive_of_binary_strings(paths, datas).get_ok()
    l1 = ctx.launches
    b = zipc.archive_of_binary_strings(paths[::-1], datas[::-1]).get_ok()
    l2 = ctx.launches
    assert bytes(a) == bytes(b)
    assert (l1 - l0) > (l2 - l1)          # the pipelined call launched one set of kernels per group
    zf = zipfile.ZipFile(io.BytesIO(bytes(a)))
    assert zf.testzip() is None and len(zf.namelist()) == n
    for i in (0, 1, n // 2, n - 1):
        assert zf.read(paths[i]) == datas[i].tobytes()


def test_zip64_archives_extract_and_create(ctx):
    """SURVEY.md 8f-4 (beyond the reference, checked against CPython's zipfile): members of a ZIP64 archive made by CPython
    are extracted on the GPU; an archive of GPU-deflated members written with ZIP64 records is read back by CPython."""
    n_small = 66_000  # more than 65,535 members: ZIP64 end of central directory record
    datas = {("big/%03d.txt" % i): synth.text_v1(500 + i, 30_000 + 1111 * i).tobytes() for i in range(24)}
    bio = io.BytesIO()
    with zipfile.ZipFile(bio, "w", zipfile.ZIP_DEFLATED) as zf:
        for i in range(n_small):
            zf.writestr("s/%05d" % i, b"%d" % i, compress_type=zipfile.ZIP_STORED)
        for p, d in datas.items():
            with zf.open(p, "w", force_zip64=True) as fh:
                fh.write(d)
    blob = bio.getvalue()
    z = zipc.of_binary_string(blob, zip64=True).get_ok()
    assert zipc.member_count(z) == n_small + len(datas)
    paths = sorted(z)
    got = zipc.File.to_binary_strings([z[p].kind for p in paths])
    for p, r in zip(paths, got):
        want = datas[p.decode()] if p.startswith(b"big/") else b"%d" % int(p[2:])
        assert r.get_ok() == want
    # the other direction
    files = zipc.File.deflate_of_binary_strings(list(datas.values()), "default")
    ours = {p.encode(): zipc.Member.make(p, f.get_ok()).get_ok() for p, f in zip(datas, files)}
    forced = zipc.to_binary_string(ours, zip64="force").get_ok()
    with zipfile.ZipFile(io.BytesIO(forced)) as zf:
        assert zf.testzip() is None
        for p, d in datas.items():
            assert zf.read(p) == d
    back = zipc.of_binary_string(forced, zip64=True).get_ok()
    for p, r in zip(sorted(back), zipc.File.to_binary_strings([back[p].kind for p in sorted(back)])):
        assert r.get_ok() == datas[p.decode()]


def test_archive_creation_with_more_than_65535_members(ctx):
    """zipc_b200_zip_deflate_archive_ex with ZIP64 allowed: one call compresses 66,000 payloads and writes the archive with a
    ZIP64 end of central directory record (the reference's call refuses: zipc.ml:574); CPython reads it."""
    n = 66_000
    paths = ["d/%05d.txt" % i for i in range(n)]
    payloads = [b"payload %d " % i * (1 + i % 7) for i in range(n)]
    r = zipc.archive_of_binary_strings(paths, payloads, "fast")
    assert r.is_error() and r.status == 28
    blob = zipc.archive_of_binary_strings(paths, payloads, "fast", zip64=True).get_ok()
    with zipfile.ZipFile(io.BytesIO(blob)) as zf:
        assert len(zf.namelist()) == n
        for i in (0, 1, 4999, 65_535, 65_999):
            assert zf.read(paths[i]) == payloads[i]
    z = zipc.of_binary_string(blob, zip64=True).get_ok()
    assert zipc.member_count(z) == n
