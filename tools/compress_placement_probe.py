#!/usr/bin/env python
"""The compress calls whose output goes through the placement gather (zip_api.cu place_pieces): what they return, and what
they cost where a host-side step would show.

--hashes FILE  For fixed seeded inputs, one line per output or status array: "<call> <array> <sha256>".  Two builds of the
               library (ZIPC_B200_LIB selects one) compute the same thing when their files are equal.
                 deflate_batch             a small batch (levels none..best, CRC-32 and Adler-32) and a batch large enough
                                           to be pipelined (1,100 members, 104 MiB)
                 zlib_compress_batch(_dev) levels none..best, both Adler-32 modes, two members above the split threshold;
                                           the _dev form at odd slot offsets, one slot too small, slots pre-filled
                 deflate_segmented/primed  last_piece 0 and 1, an empty input; stream, index and CRC-32
                 zip_deflate_archive_ex    the large batch in path order (pipelined) and in reverse order (plain path); a
                                           small set with a duplicate path and `first`, ZIP64 forced and not
                 zip_deflate_archive_dev   mixed stored and deflated members, a duplicate path, at an odd offset
--timing FILE  Host clock around calls that end in a synchronise, shapes bench.py does not time:
                 plain archive  the bench's 10,000 C3/C4 members (text-v1, 4-256 KiB) in reverse path order through
                                zip_deflate_archive_ex from pinned host memory: the plain host path
                 small calls    one 4 KiB text member through deflate_batch, zlib_compress_batch and deflate_segmented
               One warm-up, then --reps rounds; a round of the small calls is 200 calls of each.  The card's name and power
               limit are read in the same run.

  python tools/compress_placement_probe.py --hashes out.txt
  python tools/compress_placement_probe.py --timing out.txt [--reps 5]
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from zipc_b200 import _lib, synth  # noqa: E402
from zipc_b200 import zipc_deflate as zd  # noqa: E402

SZ, U32, I32 = C.c_size_t, C.c_uint32, C.c_int


def arr(t, v):
    return (t * max(len(v), 1))(*v)


def sha(x) -> str:
    if isinstance(x, C.Array):
        x = bytes(x)
    elif isinstance(x, np.ndarray):
        x = x.tobytes()
    elif isinstance(x, int):
        x = str(x).encode()
    return hashlib.sha256(x).hexdigest()


class Probe:
    def __init__(self):
        self.ctx = zd.Context(0)
        self.L, self.h = self.ctx.L, self.ctx.h
        self.lines = []

    def put(self, call, **arrays):
        for k, v in arrays.items():
            self.lines.append(f"{call} {k} {sha(v)}")

    def host(self, items):
        ptrs = arr(C.c_void_p, [x.ctypes.data if x.size else None for x in items])
        return ptrs, arr(SZ, [x.size for x in items])

    def dev(self, nbytes, fill=None):
        p = C.c_void_p()
        assert self.L.zipc_b200_dev_alloc(self.h, max(nbytes, 1), C.byref(p)) == 0
        if fill is not None:
            assert self.L.zipc_b200_memcpy_h2d(self.h, p, fill.ctypes.data, fill.size) == 0
        return p

    def read(self, p, nbytes):
        out = np.empty(max(nbytes, 1), dtype=np.uint8)
        assert self.L.zipc_b200_memcpy_d2h(self.h, out.ctypes.data, p, nbytes) == 0
        return out[:nbytes]

    # ---- the calls -------------------------------------------------------------------------------------------------
    def deflate_batch(self, name, items, level, ck, adler_mode=0):
        n = len(items)
        ptrs, lens = self.host(items)
        cap = sum((self.L.zipc_b200_deflate_bound(x.size) + 15) & ~15 for x in items) + 4096
        dst = np.zeros(cap, dtype=np.uint8)
        need, off, ln, cs, st = SZ(), arr(SZ, [0] * n), arr(SZ, [0] * n), arr(U32, [0] * n), arr(I32, [0] * n)
        rc = self.L.zipc_b200_deflate_batch(self.h, level, ck, adler_mode, n, ptrs, lens, dst.ctypes.data, cap, C.byref(need),
                                            off, ln, cs, st)
        self.put(name, rc=rc, need=need.value, arena=dst[:need.value], off=off, len=ln, checksum=cs, status=st)

    def zlib_host(self, name, items, level, adler_mode):
        n = len(items)
        ptrs, lens = self.host(items)
        cap = sum((self.L.zipc_b200_zlib_bound(x.size) + 15) & ~15 for x in items) + 4096
        dst = np.zeros(cap, dtype=np.uint8)
        need, off, ln, ad, st = SZ(), arr(SZ, [0] * n), arr(SZ, [0] * n), arr(U32, [0] * n), arr(I32, [0] * n)
        rc = self.L.zipc_b200_zlib_compress_batch(self.h, level, adler_mode, n, ptrs, lens, dst.ctypes.data, cap, C.byref(need),
                                                  off, ln, ad, st)
        self.put(name, rc=rc, need=need.value, arena=dst[:need.value], off=off, len=ln, adler=ad, status=st)

    def zlib_dev(self, name, items, level, adler_mode, small=()):
        """inputs back to back at an odd offset; slot i of zlib_bound (5 bytes for i in small) at odd offsets, pre-filled"""
        n = len(items)
        src = np.concatenate([np.zeros(3, np.uint8)] + list(items))
        soff = np.concatenate([[3], 3 + np.cumsum([x.size for x in items])[:-1]]).astype(np.int64).tolist()
        caps = [5 if i in small else self.L.zipc_b200_zlib_bound(x.size) for i, x in enumerate(items)]
        doff = np.concatenate([[1], 1 + np.cumsum([c + 7 for c in caps])[:-1]]).astype(np.int64).tolist()
        total = doff[-1] + caps[-1] + 64
        fill = np.random.default_rng(5).integers(0, 256, total, dtype=np.uint8)
        ds, dd = self.dev(src.size, src), self.dev(total, fill)
        ln, ad, st = arr(SZ, [0] * n), arr(U32, [0] * n), arr(I32, [0] * n)
        rc = self.L.zipc_b200_zlib_compress_batch_dev(self.h, level, adler_mode, n, ds, arr(SZ, soff), arr(SZ, [x.size for x in items]),
                                                      dd, arr(SZ, doff), arr(SZ, caps), ln, ad, st)
        self.put(name, rc=rc, slots=self.read(dd, total), len=ln, adler=ad, status=st)
        self.L.zipc_b200_dev_free(self.h, ds)
        self.L.zipc_b200_dev_free(self.h, dd)

    def segmented(self, name, data, level, seg, last_piece, primed):
        nmax = max(1, -(-data.size // seg)) + 1
        dst = np.zeros(data.size + 6 * nmax + 4096, dtype=np.uint8)
        index = np.zeros(2 * nmax, dtype=np.uint64)
        n, nseg, crc = SZ(), SZ(), U32()
        fn = self.L.zipc_b200_deflate_primed if primed else self.L.zipc_b200_deflate_segmented
        rc = fn(self.h, level, data.ctypes.data if data.size else None, data.size, seg, last_piece, dst.ctypes.data, dst.size,
                C.byref(n), index.ctypes.data_as(C.POINTER(C.c_uint64)), nmax, C.byref(nseg), C.byref(crc))
        self.put(name, rc=rc, stream=dst[:n.value], index=index[:2 * nseg.value + 2], nseg=nseg.value, crc=crc.value)

    def archive_host(self, name, paths, items, flags=0, first=None, out=None):
        n = len(items)
        keep = [C.create_string_buffer(p, max(len(p), 1)) for p in paths]
        pp = arr(C.c_void_p, [C.cast(b, C.c_void_p).value for b in keep])
        pl = arr(U32, [len(p) for p in paths])
        ptrs, lens = self.host(items)
        if out is None:
            out = np.zeros(self.L.zipc_b200_zip_archive_bound(n, pl, lens, None), dtype=np.uint8)
        olen = SZ()
        l0 = self.ctx.launches
        rc = self.L.zipc_b200_zip_deflate_archive_ex(self.h, 2, n, pp, pl, ptrs, lens, None, None, first, flags, out.ctypes.data,
                                                     out.size, C.byref(olen))
        self.put(name, rc=rc, out_len=olen.value, archive=out[:olen.value])
        return self.ctx.launches - l0

    def archive_dev(self, name, paths, items, comp, flags=0, first=None):
        n = len(items)
        keep = [C.create_string_buffer(p, max(len(p), 1)) for p in paths]
        pp = arr(C.c_void_p, [C.cast(b, C.c_void_p).value for b in keep])
        pl = arr(U32, [len(p) for p in paths])
        lens = arr(SZ, [x.size for x in items])
        src = np.concatenate(list(items))
        soff = np.concatenate([[0], np.cumsum([x.size for x in items])[:-1]]).astype(np.int64).tolist()
        cm = arr(C.c_int32, comp)
        cap = self.L.zipc_b200_zip_archive_bound(n, pl, lens, cm)
        fill = np.random.default_rng(6).integers(0, 256, cap + 64, dtype=np.uint8)
        ds, dd = self.dev(src.size, src), self.dev(cap + 64, fill)
        olen = SZ()
        rc = self.L.zipc_b200_zip_deflate_archive_dev(self.h, 2, n, pp, pl, ds, arr(SZ, soff), lens, cm, None, None, first, flags,
                                                      C.c_void_p(dd.value + 3), cap, C.byref(olen))
        self.put(name, rc=rc, out_len=olen.value, buffer=self.read(dd, cap + 64))
        self.L.zipc_b200_dev_free(self.h, ds)
        self.L.zipc_b200_dev_free(self.h, dd)


def small_set():
    """64 members of 0 - 300 KiB, text and random, two of 3 MiB / 2.5 MiB (split: the batch is thin)"""
    rng = np.random.default_rng(11)
    items = []
    for i in range(64):
        size = int(rng.integers(0, 300 << 10)) if i % 9 else int(rng.integers(0, 300))
        items.append(synth.rand_v1(100 + i, size) if i % 7 == 3 else synth.text_v1(100 + i, size))
    items[5] = synth.text_v1(7, 3 << 20)
    items[40] = synth.text_v1(8, (5 << 19) + 12345)
    return items


def large_set():
    """1,100 text members of 64 - 128 KiB (104 MiB): pipelined by deflate_batch and by the archive call in path order"""
    rng = np.random.default_rng(12)
    return [synth.text_v1(2000 + i, int(rng.integers(64 << 10, 128 << 10))) for i in range(1100)]


def hashes(args):
    p = Probe()
    small, large = small_set(), large_set()
    for level in range(4):
        for ck in (_lib.CK_CRC32, _lib.CK_ADLER32):
            p.deflate_batch(f"deflate_batch/small/level{level}/ck{ck}", small, level, ck)
    p.deflate_batch("deflate_batch/large/level2/crc32", large, 2, _lib.CK_CRC32)
    for level in range(4):
        for mode in (_lib.ADLER_REF_COMPAT, _lib.ADLER_RFC1950):
            p.zlib_host(f"zlib_compress_batch/level{level}/adler{mode}", small, level, mode)
            p.zlib_dev(f"zlib_compress_batch_dev/level{level}/adler{mode}", small, level, mode, small=(9, 40))
    text = synth.text_v1(21, (5 << 20) + 777)
    for primed in (False, True):
        for seg in (256 << 10, 100_000):
            for last in (0, 1):
                p.segmented(f"deflate_{'primed' if primed else 'segmented'}/seg{seg}/last{last}", text, 2, seg, last, primed)
        p.segmented(f"deflate_{'primed' if primed else 'segmented'}/empty", np.zeros(0, np.uint8), 2, 4096, 1, primed)
    paths = [b"big/%05d.txt" % i for i in range(len(large))]
    big = np.zeros(sum(x.size for x in large) // 2 + 256 * len(large) + 65536, dtype=np.uint8)
    la = p.archive_host("zip_deflate_archive_ex/pipelined", paths, large, out=big)
    lb = p.archive_host("zip_deflate_archive_ex/plain_reverse", paths[::-1], large[::-1], out=big)
    print(f"archive launches: path order {la}, reverse order {lb}", flush=True)
    assert la > lb, "the path-order archive did not take the pipelined path"
    sp = [b"dir\\m%02d.txt" % i for i in range(len(small))]
    sp[10], sp[30] = b"mimetype", sp[20]
    for flags in (0, 2):
        p.archive_host(f"zip_deflate_archive_ex/small/flags{flags}", sp, small, flags=flags)
        p.archive_host(f"zip_deflate_archive_ex/small_first/flags{flags}", sp, small, flags=flags, first=b"dir/m03.txt")
        comp = [0 if i % 3 == 1 else 8 for i in range(len(small))]
        p.archive_dev(f"zip_deflate_archive_dev/mixed/flags{flags}", sp, small, comp, flags=flags)
    with open(args.hashes, "w") as f:
        f.write("\n".join(p.lines) + "\n")
    print(f"{len(p.lines)} hashes -> {args.hashes}")


def timing(args):
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True, check=True).stdout.strip()
    p = Probe()
    L, h = p.L, p.h
    out_file = open(args.timing, "w")

    def emit(line):
        print(line, flush=True)
        out_file.write(line + "\n")
        out_file.flush()
    emit(f"# card: {card}")
    emit(f"# library: {os.environ.get('ZIPC_B200_LIB') or 'in-tree'}")

    def pinned(nbytes):
        q = C.c_void_p()
        assert L.zipc_b200_host_alloc(max(nbytes, 1), C.byref(q)) == 0
        return np.ctypeslib.as_array(C.cast(q, C.POINTER(C.c_uint8)), shape=(max(nbytes, 1),))

    def rounds(fn, calls=1):
        fn()
        ts = []
        for _ in range(args.reps):
            t0 = time.perf_counter()
            for _ in range(calls):
                fn()
            ts.append((time.perf_counter() - t0) / calls)
        return ts

    # plain archive path: the 10,000 C3/C4 members in reverse path order
    sizes = synth.member_sizes(10000, seed=3)
    datas = [synth.text_v1(1000 + i, int(s)) for i, s in enumerate(sizes)][::-1]
    names = [b"m/%05d.txt" % i for i in range(10000)][::-1]
    U = int(sum(d.size for d in datas))
    src = pinned(U)
    offs = np.concatenate([[0], np.cumsum([d.size for d in datas])[:-1]]).astype(np.int64)
    for o, d in zip(offs, datas):
        src[o:o + d.size] = d
    keep = [C.create_string_buffer(x, len(x)) for x in names]
    pp = arr(C.c_void_p, [C.cast(b, C.c_void_p).value for b in keep])
    pl = arr(U32, [len(x) for x in names])
    ptrs = arr(C.c_void_p, [src.ctypes.data + int(o) for o in offs])
    lens = arr(SZ, [d.size for d in datas])
    out = pinned(U // 2 + 256 * len(datas) + 65536)
    olen = SZ()

    def create():
        assert L.zipc_b200_zip_deflate_archive_ex(h, 2, len(datas), pp, pl, ptrs, lens, None, None, None, 0, out.ctypes.data,
                                                  out.size, C.byref(olen)) == 0
    ts = rounds(create)
    emit(f"plain archive, 10000 members reverse order, {U} B in: ms " + " ".join(f"{t * 1e3:.2f}" for t in ts) +
                 f"  GB/s {U / max(ts) / 1e9:.2f}-{U / min(ts) / 1e9:.2f}")

    # one 4 KiB member
    one = synth.text_v1(77, 4096)
    s1 = pinned(4096)
    s1[:] = one
    sp, sl = arr(C.c_void_p, [s1.ctypes.data]), arr(SZ, [4096])
    d1 = pinned(1 << 16)
    need, off, ln, ck, st = SZ(), arr(SZ, [0]), arr(SZ, [0]), arr(U32, [0]), arr(I32, [0])
    idx = np.zeros(4, dtype=np.uint64)
    nseg = SZ()
    small = {
        "deflate_batch": lambda: L.zipc_b200_deflate_batch(h, 2, _lib.CK_CRC32, 0, 1, sp, sl, d1.ctypes.data, d1.size, C.byref(need),
                                                           off, ln, ck, st),
        "zlib_compress_batch": lambda: L.zipc_b200_zlib_compress_batch(h, 2, 0, 1, sp, sl, d1.ctypes.data, d1.size, C.byref(need),
                                                                       off, ln, ck, st),
        "deflate_segmented": lambda: L.zipc_b200_deflate_segmented(h, 2, s1.ctypes.data, 4096, 4096, 1, d1.ctypes.data, d1.size,
                                                                   C.byref(need), idx.ctypes.data_as(C.POINTER(C.c_uint64)), 2,
                                                                   C.byref(nseg), ck),
    }
    for k, fn in small.items():
        assert fn() == 0
        ts = rounds(lambda: fn(), calls=200)
        emit(f"one 4 KiB member, {k}: us/call " + " ".join(f"{t * 1e6:.1f}" for t in ts))
    out_file.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--hashes")
    ap.add_argument("--timing")
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    if args.hashes:
        hashes(args)
    if args.timing:
        timing(args)


if __name__ == "__main__":
    main()
