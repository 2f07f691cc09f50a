#!/usr/bin/env python
"""Device-resident ZIP extraction on three archive shapes: zipc_b200_zip_parse_dev and zipc_b200_zip_extract_batch_dev with
the archive and the outputs in device memory, the stored-member kernel's share of the HBM peak, and the host-pointer
zipc_b200_zip_extract_batch end to end from pinned host memory, this build against another build of the library (--parent-lib,
e.g. the parent commit's) loaded into the same process.

Shapes:
  deflate     the benchmark's 10,000 C3/C4 members (text-v1, 4-256 KiB, bench.py make_members sizes) deflated into one archive
              by this library at level default
  checkpoint  a torch.save archive of about 2 GiB: --tensors uint8 tensors of equal size plus torch's small pickle members
  stored      the same 10,000 C3 payloads as stored members (CPython zipfile, ZIP_STORED)

Device calls are bracketed by CUDA events on the context's stream; the host-pointer calls, which return only when their output
is in the caller's pinned arena, by the host clock.  Each call is made once to warm up, then the calls alternate, --reps runs
each.  The stored kernel's time comes from the library's own events around it (zipc_b200_ctx_profile).  All inputs are
larger than the 126 MB L2.  The card's name and power limit are read in the same run.

  python tools/zip_dev_probe.py [--parent-lib path/libzipc_b200.so] [--out profiles/r05_zip_dev.txt]
"""
from __future__ import annotations

import argparse
import ctypes as C
import io
import json
import os
import subprocess
import sys
import time
import zipfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def hbm_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs"
    except (OSError, KeyError, ValueError):
        return 6532.2, "DESIGN.md section 6 (MEASURED_PEAKS.json not found)"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--members", type=int, default=10000)
    ap.add_argument("--tensors", type=int, default=12)
    ap.add_argument("--checkpoint-gib", type=float, default=2.0)
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r05_zip_dev.txt"))
    args = ap.parse_args()

    import torch
    from zipc_b200 import _lib, synth, zipc
    from zipc_b200 import zipc_deflate as zd

    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True, check=True).stdout.strip()
    torch.cuda.set_device(0)
    ctx = zd.Context(0)
    zd.set_default_context(ctx)
    L, h = ctx.L, ctx.h
    stream = torch.cuda.ExternalStream(ctx.stream)
    peak, peak_src = hbm_peak()

    parent = None
    if args.parent_lib:
        PL = C.CDLL(os.path.abspath(args.parent_lib))   # (declared here: an older build lacks the newer exports)
        vp, sz, P = C.c_void_p, C.c_size_t, C.POINTER
        for name, res, argt in (("zipc_b200_ctx_create", C.c_int, [C.c_int, P(vp)]), ("zipc_b200_ctx_destroy", None, [vp]),
                                ("zipc_b200_free", None, [vp]),
                                ("zipc_b200_zip_parse_ex", C.c_int, [vp, sz, C.c_uint, P(P(_lib.Member)), P(sz)]),
                                ("zipc_b200_zip_extract_batch", C.c_int, [vp, P(_lib.Member), sz, vp, sz, P(sz), P(sz), P(sz),
                                                                          P(C.c_uint32), P(C.c_int)])):
            getattr(PL, name).restype, getattr(PL, name).argtypes = res, argt
        ph = C.c_void_p()
        assert PL.zipc_b200_ctx_create(0, C.byref(ph)) == _lib.OK
        parent = (PL, ph.value)

    # ---- the three archives ----------------------------------------------------------------------------------------------
    n = args.members
    sizes = [int(s) for s in synth.member_sizes(n, seed=3)]
    payloads = [synth.text_v1(1000 + i, m).tobytes() for i, m in enumerate(sizes)]
    names = ["m/%05d.txt" % i for i in range(n)]
    shapes = {}
    shapes["deflate"] = zipc.archive_of_binary_strings(names, payloads, "default").get_ok()
    per = int(args.checkpoint_gib * (1 << 30)) // args.tensors
    g = torch.Generator().manual_seed(9)
    sd = {"layer%02d.weight" % k: torch.randint(0, 256, (per,), generator=g, dtype=torch.uint8) for k in range(args.tensors)}
    bio = io.BytesIO()
    torch.save(sd, bio)
    del sd
    shapes["checkpoint"] = bio.getvalue()
    del bio
    bio = io.BytesIO()
    with zipfile.ZipFile(bio, "w", zipfile.ZIP_STORED) as zf:
        for nm, p in zip(names, payloads):
            zf.writestr(nm, p)
    shapes["stored"] = bio.getvalue()
    del bio, payloads

    def alloc(nbytes):
        p = C.c_void_p()
        ctx._check(L.zipc_b200_dev_alloc(h, nbytes, C.byref(p)), "dev_alloc")
        return p.value

    def halloc(nbytes):
        p = C.c_void_p()
        ctx._check(L.zipc_b200_host_alloc(nbytes, C.byref(p)), "host_alloc")
        return p.value

    def events(fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record(stream)
        fn()
        b.record(stream)
        torch.cuda.synchronize()
        return a.elapsed_time(b)

    def wall(fn):
        t0 = time.perf_counter()
        fn()
        return (time.perf_counter() - t0) * 1e3

    lines = ["# tools/zip_dev_probe.py: device-resident ZIP parse and extraction, and the host-pointer extraction of two builds",
             f"# card: {card} (nvidia-smi name, power.limit, read in this run)",
             f"# HBM peak for the stored kernel's share: {peak:.1f} GB/s ({peak_src})",
             "# parse_dev / extract_batch_dev: CUDA events on the context's stream around the call, archive and outputs in device",
             "#   memory (zipc_b200_dev_alloc), output slots back to back; stored kernel: the library's events around it",
             "# extract_batch (host): host clock around the call, archive and arena in pinned host memory (zipc_b200_host_alloc)",
             f"# one warm-up call each, then the calls alternate, {args.reps} runs each; GB/s = extracted bytes / time", ""]

    for shape, data in shapes.items():
        A = len(data)
        host_arch = halloc(A)
        C.memmove(host_arch, data, A)
        d_arch = alloc(A)
        ctx._check(L.zipc_b200_memcpy_h2d(h, d_arch, host_arch, A), "memcpy_h2d")
        del data
        # device members
        p, cnt = C.POINTER(_lib.Member)(), C.c_size_t()
        ctx._check(L.zipc_b200_zip_parse_dev(h, d_arch, A, 0, C.byref(p), C.byref(cnt)), "zip_parse_dev")
        m = cnt.value
        caps = [0 if p[i].is_dir else (p[i].compressed_size if p[i].compression == 0 else p[i].decompressed_size) for i in range(m)]
        stored_bytes = sum(caps[i] for i in range(m) if not p[i].is_dir and p[i].compression == 0)
        U = sum(caps)
        doff = np.concatenate([[0], np.cumsum(caps)[:-1]]).astype(np.int64) if m else np.zeros(0, np.int64)
        d_out = alloc(U + 64)
        dl, fo, st = (C.c_size_t * m)(), (C.c_uint32 * m)(), (C.c_int * m)()
        do = (C.c_size_t * m)(*[int(x) for x in doff])

        def parse_dev():
            q, c2 = C.POINTER(_lib.Member)(), C.c_size_t()
            ctx._check(L.zipc_b200_zip_parse_dev(h, d_arch, A, 0, C.byref(q), C.byref(c2)), "zip_parse_dev")
            L.zipc_b200_free(C.cast(q, C.c_void_p))

        def extract_dev():
            ctx._check(L.zipc_b200_zip_extract_batch_dev(h, p, m, d_out, do, dl, fo, st), "zip_extract_batch_dev")
            bad = [i for i in range(m) if st[i] != _lib.OK]
            assert not bad, f"{shape}: member {bad[0]} status {st[bad[0]]}"

        # host-pointer extraction, per build: members parsed from the pinned archive, outputs into a pinned arena
        hosts = [("new", L, h)] + ([("parent", parent[0], parent[1])] if parent else [])
        harena = halloc(U + 16 * m + 64)
        hcalls = {}
        for tag, LL, hh in hosts:
            hp, hc = C.POINTER(_lib.Member)(), C.c_size_t()
            assert LL.zipc_b200_zip_parse_ex(host_arch, A, 0, C.byref(hp), C.byref(hc)) == _lib.OK
            need = C.c_size_t()
            hoff, hln = (C.c_size_t * m)(), (C.c_size_t * m)()
            hfo, hst = (C.c_uint32 * m)(), (C.c_int * m)()

            def call(LL=LL, hh=hh, hp=hp, need=need, hoff=hoff, hln=hln, hfo=hfo, hst=hst):
                rc = LL.zipc_b200_zip_extract_batch(hh, hp, m, harena, U + 16 * m + 64, C.byref(need), hoff, hln, hfo, hst)
                assert rc == _lib.OK, rc
                assert all(hst[i] == _lib.OK for i in range(m))
            hcalls[tag] = (call, hp, LL)

        L.zipc_b200_ctx_profile(h, 1)
        order = [("parse_dev", lambda: events(parse_dev)), ("extract_batch_dev", lambda: events(extract_dev))]
        order += [(f"extract_batch host {tag}", (lambda c=c: wall(c))) for tag, (c, _, _) in hcalls.items()]
        ms = {k: [] for k, _ in order}
        kern = []
        for k, fn in order:
            fn()
        for _ in range(args.reps):
            for k, fn in order:
                ms[k].append(fn())
                if k == "extract_batch_dev":
                    kern.append(L.zipc_b200_ctx_kernel_ms(h))
        L.zipc_b200_ctx_profile(h, 0)
        # the device outputs are the host call's: compare a sample of members byte for byte
        out = np.empty(U + 64, dtype=np.uint8)
        ctx._check(L.zipc_b200_memcpy_d2h(h, out.ctypes.data, d_out, U + 64), "memcpy_d2h")
        hv = np.ctypeslib.as_array((C.c_uint8 * (U + 16 * m + 64)).from_address(harena))
        call, hp, _ = hcalls["new"]
        need = C.c_size_t()
        hoff, hln, hfo, hst = (C.c_size_t * m)(), (C.c_size_t * m)(), (C.c_uint32 * m)(), (C.c_int * m)()
        assert L.zipc_b200_zip_extract_batch(h, hp, m, harena, U + 16 * m + 64, C.byref(need), hoff, hln, hfo, hst) == _lib.OK
        for i in range(0, m, max(1, m // 97)):
            assert dl[i] == hln[i] and fo[i] == hfo[i], (shape, i)
            assert (out[doff[i]:doff[i] + dl[i]] == hv[hoff[i]:hoff[i] + hln[i]]).all(), (shape, i)

        lines.append(f"## {shape}: archive {A} bytes, {m} members, {U} bytes extracted ({stored_bytes} of them stored)")
        for k, _ in order:
            t = ms[k]
            rate = "" if k == "parse_dev" else f"   GB/s: {U / (max(t) / 1e3) / 1e9:.2f}-{U / (min(t) / 1e3) / 1e9:.2f}"
            lines.append(f"{k:28s} ms: " + "  ".join(f"{x:8.2f}" for x in t) + rate)
        if stored_bytes == U and U:
            bw = [2 * U / (x / 1e3) / 1e9 for x in kern]
            lines.append(f"{'stored_copy_crc_kernel':28s} ms: " + "  ".join(f"{x:8.2f}" for x in kern) +
                         f"   2N/t GB/s: {min(bw):.1f}-{max(bw):.1f} = {100 * min(bw) / peak:.1f}-{100 * max(bw) / peak:.1f} % of HBM peak")
        lines.append("")
        for tag, (_, hp_, LL) in hcalls.items():
            LL.zipc_b200_free(C.cast(hp_, C.c_void_p))
        L.zipc_b200_free(C.cast(p, C.c_void_p))
        L.zipc_b200_dev_free(h, d_arch)
        L.zipc_b200_dev_free(h, d_out)
        L.zipc_b200_host_free(host_arch)
        L.zipc_b200_host_free(harena)
        print("\n".join(lines[-(len(order) + 3):]), flush=True)

    text = "\n".join(lines)
    print(text)
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text + "\n")
    if parent:
        parent[0].zipc_b200_ctx_destroy(parent[1])
    zd.set_default_context(None)
    ctx.close()


if __name__ == "__main__":
    main()
