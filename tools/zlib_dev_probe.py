#!/usr/bin/env python
"""What the zlib framing costs on the device-resident path: zipc_b200_zlib_compress_batch_dev against
zipc_b200_deflate_batch_dev (Adler-32 of the input, level default), and zipc_b200_zlib_decompress_batch_dev against
zipc_b200_inflate_batch_dev (Adler-32 of the output) on the streams they made.

Members are the benchmark's C4 members (text-v1, 4-256 KiB, sizes of bench.py make_members), packed back to back in one
device buffer (zipc_b200_dev_alloc); outputs go to slots of zipc_b200_zlib_bound.  Each call is bracketed by CUDA events on
the context's stream; the raw and the zlib call alternate, three times each, after one warm-up call of each.  The card's
name and power limit are read in the same run.

  python tools/zlib_dev_probe.py [--members 10000] [--out profiles/r04_zlib_dev.txt]
"""
from __future__ import annotations

import argparse
import ctypes as C
import os
import subprocess
import sys
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--members", type=int, default=10000)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_zlib_dev.txt"))
    args = ap.parse_args()

    import torch
    from zipc_b200 import _lib, synth
    from zipc_b200 import zipc_deflate as zd

    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True, check=True).stdout.strip()
    torch.cuda.set_device(0)
    ctx = zd.Context(0)
    L, h = ctx.L, ctx.h
    stream = torch.cuda.ExternalStream(ctx.stream)

    n = args.members
    sizes = [int(s) for s in synth.member_sizes(n, seed=3)]
    src_off = np.concatenate([[0], np.cumsum(sizes)[:-1]]).astype(np.int64)
    U = int(sum(sizes))
    host = np.empty(U, dtype=np.uint8)
    for i, (o, m) in enumerate(zip(src_off, sizes)):
        host[o:o + m] = synth.text_v1(1000 + i, m)

    def alloc(nbytes):
        p = C.c_void_p()
        ctx._check(L.zipc_b200_dev_alloc(h, nbytes, C.byref(p)), "dev_alloc")
        return p.value

    caps = [int(L.zipc_b200_zlib_bound(m)) for m in sizes]
    slot = [(c + 15) & ~15 for c in caps]
    dst_off = np.concatenate([[0], np.cumsum(slot)[:-1]]).astype(np.int64)
    d_src, d_raw, d_zlib, d_back = alloc(U + 64), alloc(int(sum(slot)) + 64), alloc(int(sum(slot)) + 64), alloc(U + 64)
    ctx._check(L.zipc_b200_memcpy_h2d(h, d_src, host.ctypes.data, U), "memcpy_h2d")

    sz = lambda v: (C.c_size_t * n)(*[int(x) for x in v])
    so, sl, do, dc, mo = sz(src_off), sz(sizes), sz(dst_off), sz(caps), sz(sizes)
    raw_len, zlib_len, out_len = (C.c_size_t * n)(), (C.c_size_t * n)(), (C.c_size_t * n)()
    ck, ex, fo, st = (C.c_uint32 * n)(), (C.c_uint32 * n)(), (C.c_uint32 * n)(), (C.c_int * n)()
    mode = _lib.ADLER_REF_COMPAT

    def check(rc, what):
        ctx._check(rc, what)
        bad = [i for i in range(n) if st[i] != _lib.OK]
        assert not bad, f"{what}: member {bad[0]} status {st[bad[0]]}"

    calls = {
        "deflate_batch_dev": lambda: check(L.zipc_b200_deflate_batch_dev(h, _lib.LEVEL_DEFAULT, _lib.CK_ADLER32, mode, n, d_src, so, sl,
                                                                         d_raw, do, dc, raw_len, ck, st), "deflate_batch_dev"),
        "zlib_compress_batch_dev": lambda: check(L.zipc_b200_zlib_compress_batch_dev(h, _lib.LEVEL_DEFAULT, mode, n, d_src, so, sl,
                                                                                     d_zlib, do, dc, zlib_len, ck, st), "zlib_compress_batch_dev"),
        "inflate_batch_dev": lambda: check(L.zipc_b200_inflate_batch_dev(h, _lib.CK_ADLER32, mode, n, d_raw, do, raw_len, d_back, so, mo,
                                                                         out_len, ck, st), "inflate_batch_dev"),
        "zlib_decompress_batch_dev": lambda: check(L.zipc_b200_zlib_decompress_batch_dev(h, mode, n, d_zlib, do, zlib_len, d_back, so, mo,
                                                                                         out_len, ex, fo, st), "zlib_decompress_batch_dev"),
    }

    def timed(name):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record(stream)
        calls[name]()
        b.record(stream)
        torch.cuda.synchronize()
        return a.elapsed_time(b)

    pairs = [("deflate_batch_dev", "zlib_compress_batch_dev"), ("inflate_batch_dev", "zlib_decompress_batch_dev")]
    ms = {k: [] for k in calls}
    for pair in pairs:
        for name in pair:          # warm-up (the inflate pair reads what the compress pair wrote)
            timed(name)
        for _ in range(args.reps):
            for name in pair:
                ms[name].append(timed(name))

    # the zlib streams are the raw streams framed: the bodies are byte for byte the same (no member is split at these sizes)
    raw_b = np.empty(int(sum(slot)), dtype=np.uint8)
    zl_b = np.empty(int(sum(slot)), dtype=np.uint8)
    ctx._check(L.zipc_b200_memcpy_d2h(h, raw_b.ctypes.data, d_raw, raw_b.size), "memcpy_d2h")
    ctx._check(L.zipc_b200_memcpy_d2h(h, zl_b.ctypes.data, d_zlib, zl_b.size), "memcpy_d2h")
    back = np.empty(U, dtype=np.uint8)
    ctx._check(L.zipc_b200_memcpy_d2h(h, back.ctypes.data, d_back, U), "memcpy_d2h")
    assert (back == host).all(), "zlib_decompress_batch_dev did not give the members back"
    for i in range(0, n, max(1, n // 64)):
        r = raw_b[dst_off[i]:dst_off[i] + raw_len[i]].tobytes()
        z = zl_b[dst_off[i]:dst_off[i] + zlib_len[i]].tobytes()
        assert z[2:-4] == r and zlib.decompress(z) == host[src_off[i]:src_off[i] + sizes[i]].tobytes(), i
    C_raw, C_zlib = int(sum(raw_len[i] for i in range(n))), int(sum(zlib_len[i] for i in range(n)))

    lines = [f"# tools/zlib_dev_probe.py --members {n}: device-resident zlib framing against the raw calls",
             f"# card: {card} (nvidia-smi name, power.limit, read in this run)",
             f"# {n} C4 members (text-v1, 4-256 KiB), {U} bytes uncompressed; level default, Adler-32 REF_COMPAT on both sides",
             f"# compressed: {C_raw} bytes raw, {C_zlib} bytes zlib (+6 per member); inputs and outputs in device memory",
             "# per call: CUDA events on the context's stream around the call; the two calls of a pair alternate, one warm-up each",
             "# GB/s = uncompressed bytes / call time", ""]
    for pair in pairs:
        for name in pair:
            t = ms[name]
            lines.append(f"{name:27s} ms: " + "  ".join(f"{x:8.2f}" for x in t) +
                         f"   GB/s: {U / (max(t) / 1e3) / 1e9:.2f}-{U / (min(t) / 1e3) / 1e9:.2f}")
        a, b = pair
        d = [y - x for x, y in zip(ms[a], ms[b])]
        lines.append(f"{'  zlib call - raw call':27s} ms: " + "  ".join(f"{x:8.2f}" for x in d) + f"   (median {float(np.median(d)):.2f} ms)")
        lines.append("")
    text = "\n".join(lines)
    print(text)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text + "\n")
    for p in (d_src, d_raw, d_zlib, d_back):
        L.zipc_b200_dev_free(h, p)
    ctx.close()


if __name__ == "__main__":
    main()
