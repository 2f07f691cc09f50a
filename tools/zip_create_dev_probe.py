#!/usr/bin/env python
"""Device-resident ZIP creation on two shapes: zipc_b200_zip_deflate_archive_dev with the payloads and the archive in
device memory.

Shapes:
  deflate     the benchmark's 10,000 C3/C4 members (text-v1, 4-256 KiB, bench.py make_members sizes) deflated at level default,
              against zipc_b200_deflate_batch_dev with CRC-32 over the same payloads into 16-byte aligned slots: the
              difference is the gather into the archive, the header kernel and one more synchronisation
  checkpoint  the members of a torch.save archive of about 2 GiB (--tensors uint8 tensors of equal size plus torch's small
              members), all stored: the stored kernel (stored_copy_crc_kernel) copies and checksums them into the archive

Calls are bracketed by CUDA events on the context's stream; the stored kernel's time comes from the library's own events
around it (zipc_b200_ctx_profile).  Each call is made once to warm up, then the calls alternate, --reps runs each.  All
inputs are larger than the 126 MB L2.  The card's name and power limit are read in the same run.  Each archive is checked once
after the timed runs: the deflate one by the host parser and zipfile, the checkpoint by torch.load.

  python tools/zip_create_dev_probe.py [--out profiles/r06_zip_create_dev.txt]
"""
from __future__ import annotations

import argparse
import ctypes as C
import io
import json
import os
import subprocess
import sys
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
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r06_zip_create_dev.txt"))
    args = ap.parse_args()

    import torch
    from zipc_b200 import _lib, synth
    from zipc_b200 import zipc_deflate as zd

    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                          capture_output=True, text=True, check=True).stdout.strip()
    torch.cuda.set_device(0)
    ctx = zd.Context(0)
    zd.set_default_context(ctx)
    L, h = ctx.L, ctx.h
    stream = torch.cuda.ExternalStream(ctx.stream)
    peak, peak_src = hbm_peak()

    def szs(v):
        return (C.c_size_t * max(len(v), 1))(*v)

    def events(fn):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        a.record(stream)
        fn()
        b.record(stream)
        torch.cuda.synchronize()
        return a.elapsed_time(b)

    def to_device(payloads):
        """the payloads back to back (no alignment) in one CUDA tensor -> tensor, offsets, lengths"""
        lens = [len(p) for p in payloads]
        offs = np.concatenate([[0], np.cumsum(lens)[:-1]]).astype(np.int64).tolist()
        host = np.empty(max(sum(lens), 1), dtype=np.uint8)
        for o, p in zip(offs, payloads):
            host[o:o + len(p)] = np.frombuffer(p, dtype=np.uint8)
        return torch.from_numpy(host).cuda(), offs, lens

    class Archive:
        """one zipc_b200_zip_deflate_archive_dev call's arguments, its output in a CUDA tensor of the bound's size"""

        def __init__(self, names, src, offs, lens, comp):
            self.n = len(names)
            self.bufs = [C.create_string_buffer(p, max(len(p), 1)) for p in names]
            self.pp = (C.c_void_p * self.n)(*[C.cast(b, C.c_void_p).value for b in self.bufs])
            self.pl = (C.c_uint32 * self.n)(*[len(p) for p in names])
            self.src, self.offs, self.lens = src, szs(offs), szs(lens)
            self.comp = None if comp is None else (C.c_int32 * self.n)(*comp)
            self.cap = L.zipc_b200_zip_archive_bound(self.n, self.pl, self.lens, self.comp)
            self.out = torch.empty(self.cap, dtype=torch.uint8, device="cuda:0")
            self.out_len = C.c_size_t()

        def __call__(self):
            ctx._check(L.zipc_b200_zip_deflate_archive_dev(h, _lib.LEVEL_DEFAULT, self.n, self.pp, self.pl, self.src.data_ptr(),
                                                           self.offs, self.lens, self.comp, None, None, None, 0,
                                                           self.out.data_ptr(), self.cap, C.byref(self.out_len)),
                       "zip_deflate_archive_dev")

        def bytes(self):
            return self.out[:self.out_len.value].cpu().numpy().tobytes()

    lines = ["# tools/zip_create_dev_probe.py: device-resident ZIP creation (zipc_b200_zip_deflate_archive_dev)",
             f"# card: {card} (nvidia-smi name, power.limit, read in this run)",
             f"# HBM peak for the stored kernel's share: {peak:.1f} GB/s ({peak_src})",
             "# CUDA events on the context's stream around each call, payloads and archive in device memory (CUDA tensors);",
             "#   stored kernel: the library's events around it",
             f"# one warm-up call each, then the calls alternate, {args.reps} runs each", ""]

    # ---- deflate: the 10,000 C3/C4 members at level default -----------------------------------------------------------
    n = args.members
    sizes = [int(s) for s in synth.member_sizes(n, seed=3)]
    payloads = [synth.text_v1(1000 + i, m).tobytes() for i, m in enumerate(sizes)]
    names = [b"m/%05d.txt" % i for i in range(n)]
    src, offs, lens = to_device(payloads)
    U = sum(lens)
    arch = Archive(names, src, offs, lens, None)
    caps = [(L.zipc_b200_deflate_bound(x) + 15) & ~15 for x in lens]
    soffs = np.concatenate([[0], np.cumsum(caps)[:-1]]).astype(np.int64).tolist()
    slots = torch.empty(sum(caps), dtype=torch.uint8, device="cuda:0")
    dl, ck, st = (C.c_size_t * n)(), (C.c_uint32 * n)(), (C.c_int * n)()
    c_offs, c_lens, c_soffs, c_caps = szs(offs), szs(lens), szs(soffs), szs(caps)

    def deflate_dev():
        ctx._check(L.zipc_b200_deflate_batch_dev(h, _lib.LEVEL_DEFAULT, _lib.CK_CRC32, 0, n, src.data_ptr(), c_offs, c_lens,
                                                 slots.data_ptr(), c_soffs, c_caps, dl, ck, st), "deflate_batch_dev")
        assert all(st[i] == _lib.OK for i in range(n))

    order = {"zip_deflate_archive_dev": arch, "deflate_batch_dev CRC-32": deflate_dev}
    times = {k: [] for k in order}
    for fn in order.values():
        events(fn)
    for _ in range(args.reps):
        for k, fn in order.items():
            times[k].append(events(fn))
    data = arch.bytes()
    zf = zipfile.ZipFile(io.BytesIO(data))
    assert zf.testzip() is None and len(zf.infolist()) == n
    crcs = {i.filename: i.CRC for i in zf.infolist()}
    assert all(crcs["m/%05d.txt" % i] == ck[i] for i in range(n))
    lines.append(f"## deflate: {n} members, {U} bytes in, archive {len(data)} bytes (level default)")
    for k, t in times.items():
        lines.append(f"{k:28s} ms: " + "  ".join(f"{x:8.2f}" for x in t) +
                     f"   GB/s in: {U / max(t) / 1e6:.2f}-{U / min(t) / 1e6:.2f}")
    lines.append("")
    print("\n".join(lines[-(len(order) + 2):]), flush=True)
    del arch, slots, src, payloads, data, zf

    # ---- checkpoint: the members of a torch.save archive, stored ------------------------------------------------------
    per = int(args.checkpoint_gib * (1 << 30)) // args.tensors
    g = torch.Generator().manual_seed(9)
    sd = {"layer%02d.weight" % k: torch.randint(0, 256, (per,), generator=g, dtype=torch.uint8) for k in range(args.tensors)}
    bio = io.BytesIO()
    torch.save(sd, bio)
    zf = zipfile.ZipFile(io.BytesIO(bio.getvalue()))
    del bio
    names = [i.filename.encode() for i in zf.infolist()]
    payloads = [zf.read(i) for i in zf.infolist()]
    del zf
    src, offs, lens = to_device(payloads)
    del payloads
    U = sum(lens)
    arch = Archive(names, src, offs, lens, [0] * len(names))
    arch()
    L.zipc_b200_ctx_profile(h, 1)
    t_call, t_kern = [], []
    for _ in range(args.reps):
        t_call.append(events(arch))
        t_kern.append(L.zipc_b200_ctx_kernel_ms(h))
    L.zipc_b200_ctx_profile(h, 0)
    back = torch.load(io.BytesIO(arch.bytes()))
    assert back.keys() == sd.keys() and all(torch.equal(back[k], sd[k]) for k in sd)
    lines.append(f"## checkpoint: {len(names)} members stored, {U} bytes in, archive {arch.out_len.value} bytes")
    lines.append(f"{'zip_deflate_archive_dev':28s} ms: " + "  ".join(f"{x:8.2f}" for x in t_call) +
                 f"   2N/t GB/s: {2 * U / max(t_call) / 1e6:.1f}-{2 * U / min(t_call) / 1e6:.1f} = "
                 f"{200 * U / max(t_call) / 1e6 / peak:.1f}-{200 * U / min(t_call) / 1e6 / peak:.1f} % of HBM peak")
    lines.append(f"{'stored_copy_crc_kernel':28s} ms: " + "  ".join(f"{x:8.2f}" for x in t_kern) +
                 f"   2N/t GB/s: {2 * U / max(t_kern) / 1e6:.1f}-{2 * U / min(t_kern) / 1e6:.1f} = "
                 f"{200 * U / max(t_kern) / 1e6 / peak:.1f}-{200 * U / min(t_kern) / 1e6 / peak:.1f} % of HBM peak")
    print("\n".join(lines[-3:]), flush=True)
    text = "\n".join(lines) + "\n"
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text)
    zd.set_default_context(None)
    ctx.close()


if __name__ == "__main__":
    main()
