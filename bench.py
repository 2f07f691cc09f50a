#!/usr/bin/env python
"""bench.py -- headline measurement of the zipc hot path on B200 (contract: DESIGN.md "Measurement").

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload deflate|inflate|crc32] [--level L] [--impl reference]
                  [--dump-outputs DIR]

One "step" is one pass of the hot path over one batch of synthetic input (SURVEY.md 8d):
  deflate (default; BASELINE.json configs[3], the first item of its metric): batch deflate + CRC-32 of 10,000
          text-v1 members of 4-256 KiB (1.33 GB) per GPU, level `Default
  inflate (configs[2]): batch inflate + CRC-32 of the same members
  crc32   (configs[1]): CRC-32 of a 1 GiB rand-v1 buffer (test_crc_speed shape)
`value` is device-resident throughput in GB/s of UNCOMPRESSED bytes (CUDA events on the library's stream, inputs
resident in HBM); `e2e` is the same metric through the C-ABI call with pinned HOST buffers, H2D and D2H inside the
timed region.  Inputs are larger than L2 (>= 1 GiB per step), so no L2 flush is needed between iterations.
With N > 1 (torchrun) every rank runs the same per-GPU workload on its own GPU (weak scaling: members / buffers are
independent units, no data-path collective); rank 0 prints the aggregate.  "also" carries, at every N, the other
workloads and levels (fewer steps), the compression ratio against the reference's (`ratio_vs_ref`), and for N > 1 a
STRONG-scaling leg: ONE member set / ONE buffer driven over all N GPUs through the library's box-wide entry points
(zipc_b200_multi_*), results gathered to the host and CRCs combined inside the timed region.

--dump-outputs DIR writes what the headline call handed back in its last timed step as DIR/<name>.npy (float64 for
statuses, sizes and CRC-32s, float32 for bytes; rank 0 only).  Inputs are seeded, so two builds run with the same
arguments can be compared output for output:
  deflate / inflate: status, crc32, compressed_size / decompressed_size of every member, and the output bytes of a fixed
                     seeded sample of members (sample_members, sample_compressed_bytes / sample_decompressed_bytes)
  crc32:             crc32 of the buffer

--impl reference times the reference's algorithm on the host cores.  The reference is OCaml and this image has no
OCaml toolchain, so it is the C restatement in oracle/ ("port").  That arm never loads libzipc_b200.so.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
import zlib
from concurrent.futures import ThreadPoolExecutor

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

GiB = 1 << 30
METRIC = {"crc32": "crc32_GBps_uncompressed", "inflate": "inflate_GBps_uncompressed", "deflate": "deflate_GBps_uncompressed"}
LEVELS = {"none": 0, "fast": 1, "default": 2, "best": 3}


def workload_desc(which, level="default", members=10000):
    return {
        "crc32": "C2: CRC-32 over a 1 GiB rand-v1(seed=2) buffer per GPU (test_crc_speed shape)",
        "inflate": f"C3: batch inflate + CRC-32 of {members} deflate members (text-v1, 4-256 KiB, 1.33 GB per 10k) per GPU",
        "deflate": f"C4: batch deflate (level {level}) + CRC-32 of {members} members (text-v1, 4-256 KiB, 1.33 GB per 10k) per GPU",
    }[which]


def make_config(which, level, members):
    """identical in both arms (the driver compares the dicts)"""
    c = {"workload": workload_desc(which, level, members), "l2": "inputs larger than L2 (>= 1 GiB per step), no flush needed"}
    if which != "crc32":
        c["members"] = members
        c["level"] = level
    return c


def ncu_capture(which):
    """What the committed ncu capture of this command says about the dominant kernel (profiles/rNN_traffic.json)."""
    for name in ("r02_traffic.json", "r01_traffic.json"):
        try:
            with open(os.path.join(ROOT, "profiles", name)) as f:
                return json.load(f)[which]
        except Exception:
            continue
    return {}


def ncu_traffic(which):
    """DRAM bytes per launch of the dominant kernel"""
    t = ncu_capture(which).get("traffic_bytes")
    return int(t) if t is not None else None


def measured_peak_gbs():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def bind_near_gpu(index: int):
    """One process per GPU: run this rank (and the library's threads it spawns) on the CPUs NVML lists as local to its GPU, so
    that the pinned buffers of the end-to-end path are first touched -- and therefore placed -- on the GPU's own NUMA node."""
    try:
        import pynvml
        pynvml.nvmlInit()
        hnd = pynvml.nvmlDeviceGetHandleByIndex(index)
        words = pynvml.nvmlDeviceGetCpuAffinity(hnd, (os.cpu_count() + 63) // 64)
        cpus = {64 * w + b for w, v in enumerate(words) for b in range(64) if (int(v) >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region."""

    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.15)
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------
# inputs
# ---------------------------------------------------------------------------------------------------
def make_members(synth, count: int, seed0: int = 1000):
    """C3/C4 members: sizes 4096 + r % 258049 (seed 3), content text-v1(seed0 + i)"""
    sizes = synth.member_sizes(count, seed=3)
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as ex:
        return list(ex.map(lambda a: synth.text_v1(seed0 + a[0], int(a[1])), enumerate(sizes)))


def make_text(synth, seed: int, n: int, piece: int = 32 << 20):
    """n bytes of text-v1 made in parallel pieces (piece k uses seed * 4096 + k)"""
    out = np.empty(n, dtype=np.uint8)
    spans = [(k, o, min(piece, n - o)) for k, o in enumerate(range(0, n, piece))]

    def fill(a):
        k, o, m = a
        out[o:o + m] = synth.text_v1(seed * 4096 + k, m)
    with ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as ex:
        list(ex.map(fill, spans))
    return out


class Harness:
    def __init__(self, device: int):
        import torch
        from zipc_b200 import zipc_deflate as zd
        self.torch, self.zd = torch, zd
        torch.cuda.set_device(device)
        self.ctx = zd.Context(device)
        self.L = self.ctx.L
        self.stream = torch.cuda.ExternalStream(self.ctx.stream)
        self.device = device
        self._pins = []

    def pinned(self, arr: np.ndarray, keep: bool = False) -> np.ndarray:
        """pinned copy of arr; released by the next free_pins() unless keep is set"""
        p = C.c_void_p()
        assert self.L.zipc_b200_host_alloc(max(arr.size, 1), C.byref(p)) == 0
        out = np.ctypeslib.as_array((C.c_uint8 * max(arr.size, 1)).from_address(p.value))[:arr.size]
        out[:] = arr
        if not keep:
            self._pins.append(p)
        return out

    def free_pins(self):
        for p in self._pins:
            self.L.zipc_b200_host_free(p)
        self._pins = []

    def timed(self, fn, steps, warmup):
        """K steps bracketed by CUDA events on the library stream -> total ms."""
        torch = self.torch
        for _ in range(warmup):
            fn()
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record(self.stream)
        for _ in range(steps):
            fn()
        b.record(self.stream)
        torch.cuda.synchronize()
        return a.elapsed_time(b)

    def kernel_ms(self, fn, steps):
        """average duration of the dominant kernel alone (events recorded by the library around it)"""
        self.L.zipc_b200_ctx_profile(self.ctx.h, 1)
        ts = []
        for _ in range(steps):
            fn()
            ts.append(self.L.zipc_b200_ctx_kernel_ms(self.ctx.h))
        self.L.zipc_b200_ctx_profile(self.ctx.h, 0)
        ts = [t for t in ts if t > 0]
        return float(np.mean(ts)) if ts else None


P = lambda a, t: a.ctypes.data_as(C.POINTER(t))

DUMP_LIMIT = 64 << 20
DUMP_MEMBERS = 48   # members whose bytes --dump-outputs writes: 48 x (256 KiB + deflate overhead) as float32 < 51 MB


def member_outputs(size_name, bytes_name, dbuf, offs, lens, ck, st):
    """What a batch call hands back: status, CRC-32 and output size of every member, and the output bytes of a fixed
    seeded sample of members, as float64 / float32 (exact: sizes < 2**53, CRC-32 < 2**32, bytes < 2**8)."""
    pick = np.sort(np.random.default_rng(0).choice(len(lens), min(len(lens), DUMP_MEMBERS), replace=False))
    sample = [dbuf[int(offs[i]):int(offs[i]) + int(lens[i])].cpu().numpy() for i in pick]
    return {"status": st.astype(np.float64), "crc32": ck.astype(np.float64), size_name: lens.astype(np.float64),
            "sample_members": pick.astype(np.float64),
            bytes_name: np.concatenate(sample).astype(np.float32) if sample else np.zeros(0, dtype=np.float32)}


def write_outputs(out_dir, arrays):
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit(f"--dump-outputs: {total} bytes, more than {DUMP_LIMIT >> 20} MB (use fewer --members)")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def _pack_device(h: Harness, items, pin=True):
    """concatenate (16-byte aligned) into one (pinned) host buffer + device copy; returns offsets"""
    offs = np.zeros(len(items), dtype=np.uint64)
    lens = np.array([len(x) for x in items], dtype=np.uint64)
    t = 0
    for i, x in enumerate(items):
        offs[i] = t
        t += (len(x) + 15) & ~15
    host = np.zeros(t + 64, dtype=np.uint8)
    for i, x in enumerate(items):
        host[int(offs[i]):int(offs[i]) + len(x)] = np.frombuffer(x, dtype=np.uint8) if not isinstance(x, np.ndarray) else x
    hp = h.pinned(host) if pin else host
    return hp, h.torch.from_numpy(hp).to(f"cuda:{h.device}"), offs, lens


# ---------------------------------------------------------------------------------------------------
# workloads (GPU arm)
# ---------------------------------------------------------------------------------------------------
def run_crc32(h: Harness, steps, warmup, rank, adler=True, dump=False):
    from zipc_b200 import synth
    n = GiB
    host = h.pinned(synth.rand_v1(2 + rank, n), keep=True)  # also the strong-scaling leg's buffer
    d = h.torch.from_numpy(host).to(f"cuda:{h.device}")
    dcrc = h.torch.zeros(4, dtype=h.torch.int32, device=f"cuda:{h.device}")
    fn = lambda: h.L.zipc_b200_crc32_dev_async(h.ctx.h, d.data_ptr(), n, dcrc.data_ptr())
    l0 = h.ctx.launches
    total_ms = h.timed(fn, steps, warmup)
    launches = (h.ctx.launches - l0) // (steps + warmup) * steps
    got = int(dcrc[0].item()) & 0xFFFFFFFF
    outputs = {"crc32": np.array([got], dtype=np.float64)} if dump else None
    kms = h.kernel_ms(fn, min(steps, 10))
    out = C.c_uint32()
    e2e_fn = lambda: h.L.zipc_b200_crc32(h.ctx.h, host.ctypes.data, n, C.byref(out))
    for _ in range(2):
        e2e_fn()
    t0 = time.perf_counter()
    esteps = max(3, min(steps, 5))
    for _ in range(esteps):
        e2e_fn()
    e2e_s = (time.perf_counter() - t0) / esteps
    assert out.value == got == zlib.crc32(host), (hex(out.value), hex(got))
    ad = {}
    if adler:  # Adler-32 over the same resident buffer (synchronous call: chunk kernel + device fold + 4-byte read back)
        for name, mode in (("ref_compat", 0), ("rfc1950", 1)):
            aout = C.c_uint32()
            afn = lambda: h.L.zipc_b200_adler32_dev(h.ctx.h, d.data_ptr(), n, mode, C.byref(aout))
            for _ in range(3):
                assert afn() == 0
            t0 = time.perf_counter()
            for _ in range(10):
                afn()
            dt = (time.perf_counter() - t0) / 10
            akms = h.kernel_ms(afn, 5)
            ad[name] = {"value": "%08x" % aout.value, "GBps_per_call": round(n / dt / 1e9, 1), "ms_per_call": round(dt * 1e3, 4),
                        "roofline_frac_per_call": round(n / dt / 1e9 / measured_peak_gbs()[0], 4), "chunk_kernel_ms": round(akms, 4) if akms else None}
        assert int(ad["rfc1950"]["value"], 16) == zlib.adler32(host), ad
    return dict(units=n, total_ms=total_ms, steps=steps, launches=launches, kernel_ms=kms, algo_bytes=n, e2e_s=e2e_s,
                h2d=n, d2h=4, host=host, kernel="crc32_tiles_kernel", extra={"crc32": "%08x" % got, "adler32": ad}, outputs=outputs)


def run_deflate(h: Harness, datas, level, steps, warmup, e2e=True, keep_streams=False, dump=False):
    from zipc_b200 import _lib
    lvl = LEVELS[level]
    n = len(datas)
    U = int(sum(d.size for d in datas))
    hsrc, dsrc, soff, slen = _pack_device(h, datas)
    cap = np.array([(h.L.zipc_b200_deflate_bound(int(x)) + 15) & ~15 for x in slen], dtype=np.uint64)
    doff = np.concatenate([[0], np.cumsum(cap)[:-1]]).astype(np.uint64)
    ddst = h.torch.empty(int(cap.sum()) + 64, dtype=h.torch.uint8, device=f"cuda:{h.device}")
    dl = np.zeros(n, dtype=np.uint64); ck = np.zeros(n, dtype=np.uint32); st = np.zeros(n, dtype=np.int32)

    def fn():
        rc = h.L.zipc_b200_deflate_batch_dev(h.ctx.h, lvl, 2, 0, n, dsrc.data_ptr(), P(soff, C.c_size_t), P(slen, C.c_size_t),
                                             ddst.data_ptr(), P(doff, C.c_size_t), P(cap, C.c_size_t), P(dl, C.c_size_t),
                                             P(ck, C.c_uint32), P(st, C.c_int))
        assert rc == 0, rc
    l0 = h.ctx.launches
    total_ms = h.timed(fn, steps, warmup)
    launches = (h.ctx.launches - l0) // (steps + warmup) * steps
    assert (st == 0).all(), "deflate status"
    outputs = member_outputs("compressed_size", "sample_compressed_bytes", ddst, doff, dl, ck, st) if dump else None
    Cb = int(dl.sum())
    sizes = dl.copy()
    # parity spot check inside the bench: CRC-32 of the input and a zlib round trip of a sample straight from the device
    for i in list(range(0, n, max(1, n // 24)))[:24]:
        assert int(ck[i]) == zlib.crc32(datas[i]), "crc parity lost in bench"
        cs = ddst[int(doff[i]):int(doff[i]) + int(dl[i])].cpu().numpy().tobytes()
        assert zlib.decompress(cs, -15) == datas[i].tobytes(), "round trip lost in bench"
    kms = h.kernel_ms(fn, min(steps, 3))
    r = dict(units=U, total_ms=total_ms, steps=steps, launches=launches, kernel_ms=kms, algo_bytes=U + Cb, kernel="deflate_kernel",
             sizes=sizes, h2d=U, d2h=Cb, e2e_s=None, outputs=outputs,
             extra={"uncompressed_bytes": U, "compressed_bytes": Cb, "ratio": round(Cb / U, 4)})
    if e2e:
        e_ptrs = (C.c_void_p * n)(*[hsrc.ctypes.data + int(o) for o in soff])
        e_arena = h.pinned(np.zeros(U // 2 + 16 * n + 4096, dtype=np.uint8))
        e_need = C.c_size_t(); e_off = np.zeros(n, dtype=np.uint64)

        def e2e_fn():
            rc = h.L.zipc_b200_deflate_batch(h.ctx.h, lvl, 2, 0, n, e_ptrs, P(slen, C.c_size_t), e_arena.ctypes.data, e_arena.size,
                                             C.byref(e_need), P(e_off, C.c_size_t), P(dl, C.c_size_t), P(ck, C.c_uint32), P(st, C.c_int))
            assert rc == 0 and (st == 0).all(), rc
        e2e_fn()
        t0 = time.perf_counter()
        esteps = max(2, min(steps, 3))
        for _ in range(esteps):
            e2e_fn()
        r["e2e_s"] = (time.perf_counter() - t0) / esteps
        if keep_streams:
            r["streams"] = [e_arena[int(e_off[i]):int(e_off[i]) + int(dl[i])].copy() for i in range(n)]
    return r


def run_inflate(h: Harness, datas, streams, steps, warmup, e2e=True, dump=False):
    n = len(datas)
    U = int(sum(d.size for d in datas)); Cb = int(sum(len(s) for s in streams))
    hcs, dcs, coff, clen = _pack_device(h, streams)
    slen = np.array([d.size for d in datas], dtype=np.uint64)
    soff = np.concatenate([[0], np.cumsum((slen + np.uint64(15)) & ~np.uint64(15))[:-1]]).astype(np.uint64)
    ddst = h.torch.empty(int(soff[-1] + slen[-1]) + 64, dtype=h.torch.uint8, device=f"cuda:{h.device}")
    dl = np.zeros(n, dtype=np.uint64); ck = np.zeros(n, dtype=np.uint32); st = np.zeros(n, dtype=np.int32)

    def fn():
        rc = h.L.zipc_b200_inflate_batch_dev(h.ctx.h, 2, 0, n, dcs.data_ptr(), P(coff, C.c_size_t), P(clen, C.c_size_t),
                                             ddst.data_ptr(), P(soff, C.c_size_t), P(slen, C.c_size_t), P(dl, C.c_size_t),
                                             P(ck, C.c_uint32), P(st, C.c_int))
        assert rc == 0, rc
    l0 = h.ctx.launches
    total_ms = h.timed(fn, steps, warmup)
    launches = (h.ctx.launches - l0) // (steps + warmup) * steps
    assert (st == 0).all() and (dl == slen).all(), "inflate status"
    outputs = member_outputs("decompressed_size", "sample_decompressed_bytes", ddst, soff, dl, ck, st) if dump else None
    for i in list(range(0, n, max(1, n // 200)))[:200]:
        assert int(ck[i]) == zlib.crc32(datas[i]), "crc parity lost in bench"
    i = n // 3
    assert ddst[int(soff[i]):int(soff[i]) + int(slen[i])].cpu().numpy().tobytes() == datas[i].tobytes()
    kms = h.kernel_ms(fn, min(steps, 3))
    r = dict(units=U, total_ms=total_ms, steps=steps, launches=launches, kernel_ms=kms, algo_bytes=U + Cb, kernel="inflate_kernel<false>",
             h2d=Cb, d2h=U, e2e_s=None, outputs=outputs, extra={"uncompressed_bytes": U, "compressed_bytes": Cb, "ratio": round(Cb / U, 4)})
    if e2e:  # compressed members inside one pinned host buffer (an in-memory archive), pinned output arena
        e_ptrs = (C.c_void_p * n)(*[hcs.ctypes.data + int(o) for o in coff])
        e_arena = h.pinned(np.zeros(int(((slen + np.uint64(15)) & ~np.uint64(15)).sum()) + 64, dtype=np.uint8))
        e_need = C.c_size_t(); e_off = np.zeros(n, dtype=np.uint64)

        def e2e_fn():
            rc = h.L.zipc_b200_inflate_batch(h.ctx.h, 2, 0, n, e_ptrs, P(clen, C.c_size_t), P(slen, C.c_size_t), e_arena.ctypes.data,
                                             e_arena.size, C.byref(e_need), P(e_off, C.c_size_t), P(dl, C.c_size_t), P(ck, C.c_uint32), P(st, C.c_int))
            assert rc == 0 and (st == 0).all(), rc
        e2e_fn()
        t0 = time.perf_counter()
        esteps = max(2, min(steps, 3))
        for _ in range(esteps):
            e2e_fn()
        r["e2e_s"] = (time.perf_counter() - t0) / esteps
    return r


def run_archive(h: Harness, datas, oracle_archive=None):
    """ZIP archive layer end to end (pinned host buffers): Zipc.File.deflate_of_binary_string x n + Zipc.to_binary_string in
    one call, then Zipc.of_binary_string + File.to_binary_string x n (CRC-32 checked); the same extraction of an archive
    made by the ORACLE (the reference's own encoder, restated) when one is given."""
    import io
    import zipfile
    from zipc_b200 import _lib
    n = len(datas)
    U = int(sum(d.size for d in datas))
    off = np.concatenate([[0], np.cumsum([d.size for d in datas])[:-1]]).astype(np.int64)
    src = h.pinned(np.concatenate(datas))
    names = [b"m/%05d.txt" % i for i in range(n)]
    paths = (C.c_void_p * n)(*[C.cast(C.c_char_p(x), C.c_void_p).value for x in names])  # `names` keeps the bytes alive
    plen = np.array([len(x) for x in names], dtype=np.uint32)
    ptrs = (C.c_void_p * n)(*[src.ctypes.data + int(o) for o in off])
    slen = np.array([d.size for d in datas], dtype=np.uint64)
    out = h.pinned(np.zeros(U // 2 + 256 * n + 65536, dtype=np.uint8))
    olen = C.c_size_t()

    def create():
        rc = h.L.zipc_b200_zip_deflate_archive(h.ctx.h, 2, n, paths, P(plen, C.c_uint32), ptrs, P(slen, C.c_size_t), None, None, None,
                                               out.ctypes.data, out.size, C.byref(olen))
        assert rc == 0, rc
    create()
    t0 = time.perf_counter(); create(); tc = time.perf_counter() - t0
    alen = olen.value
    zf = zipfile.ZipFile(io.BytesIO(bytes(out[:alen])))  # an independent reader sees the same members
    assert len(zf.namelist()) == n
    for i in (0, n // 2, n - 1):
        assert zf.read(names[i].decode()) == datas[i].tobytes()
    arena = h.pinned(np.zeros(U + 16 * n + 4096, dtype=np.uint8))
    need = C.c_size_t(); doff = np.zeros(n, dtype=np.uint64); dlen = np.zeros(n, dtype=np.uint64)
    found = np.zeros(n, dtype=np.uint32); st = np.zeros(n, dtype=np.int32)

    def extract(buf, blen):
        ms = C.POINTER(_lib.Member)(); cnt = C.c_size_t()
        rc = h.L.zipc_b200_zip_parse(buf.ctypes.data, blen, C.byref(ms), C.byref(cnt))
        assert rc == 0 and cnt.value == n, (rc, cnt.value)
        rc = h.L.zipc_b200_zip_extract_batch(h.ctx.h, ms, n, arena.ctypes.data, arena.size, C.byref(need), P(doff, C.c_size_t),
                                             P(dlen, C.c_size_t), P(found, C.c_uint32), P(st, C.c_int))
        h.L.zipc_b200_free(ms)
        assert rc == 0 and (st == 0).all(), rc
    extract(out, alen)
    t0 = time.perf_counter(); extract(out, alen); tx = time.perf_counter() - t0
    assert int(dlen.sum()) == U
    res = {"workload": "ZIP archive of the C3/C4 members (paths m/%05d.txt, default level): create = zipc_b200_zip_deflate_archive, "
                       "extract = zipc_b200_zip_parse + zipc_b200_zip_extract_batch (CRC-32 checked); pinned host buffers",
           "members": n, "uncompressed_bytes": U, "archive_bytes": int(alen),
           "create_e2e_GBps": round(U / tc / 1e9, 3), "extract_e2e_GBps": round(U / tx / 1e9, 3),
           "checked": "python zipfile lists all members and reads three of them back"}
    if oracle_archive is not None:
        oa = h.pinned(np.frombuffer(oracle_archive, dtype=np.uint8))
        extract(oa, oa.size)
        t0 = time.perf_counter(); extract(oa, oa.size); to = time.perf_counter() - t0
        k = n // 2  # members come back in path order = input order
        assert arena[int(doff[k]):int(doff[k]) + int(dlen[k])].tobytes() == datas[k].tobytes()
        res["oracle_made_archive"] = {"archive_bytes": int(oa.size), "extract_e2e_GBps": round(U / to / 1e9, 3),
                                      "note": "archive built by the oracle (reference encoder restated, level default, as written) with Zipc.to_binary_string's layout; every member inflated and CRC-checked on the GPU"}
    return res


def run_stream_c1(h: Harness):
    """C1: one 64 MiB text-v1 stream, segment-independent deflate + indexed inflate, pinned host buffers (e2e)"""
    from zipc_b200 import synth
    L = h.L
    data = h.pinned(synth.text_v1(1, 64 << 20))
    cbuf = h.pinned(np.zeros(data.size + (data.size >> 3) + 65536, dtype=np.uint8))
    obuf = h.pinned(np.zeros(data.size, dtype=np.uint8))
    res = {}
    for seg in (64 << 10, 256 << 10):
        nmax = -(-data.size // seg) + 1
        index = np.zeros((nmax + 1, 2), dtype=np.uint64)
        ip = index.ctypes.data_as(C.POINTER(C.c_uint64))
        n, nseg, crc, crc2, st, olen = C.c_size_t(), C.c_size_t(), C.c_uint32(), C.c_uint32(), C.c_int(), C.c_size_t()
        dfn = lambda: L.zipc_b200_deflate_segmented(h.ctx.h, 2, data.ctypes.data, data.size, seg, 1, cbuf.ctypes.data, cbuf.size,
                                                    C.byref(n), ip, nmax + 1, C.byref(nseg), C.byref(crc))
        ifn = lambda: L.zipc_b200_inflate_segmented(h.ctx.h, cbuf.ctypes.data, n.value, ip, nseg.value, obuf.ctypes.data, obuf.size,
                                                    C.byref(olen), C.byref(crc2), C.byref(st))
        assert dfn() == 0
        t0 = time.perf_counter()
        for _ in range(3): dfn()
        td = (time.perf_counter() - t0) / 3
        assert ifn() == 0 and st.value == 0
        t0 = time.perf_counter()
        for _ in range(3): ifn()
        ti = (time.perf_counter() - t0) / 3
        assert crc2.value == crc.value and olen.value == data.size and bytes(obuf[:4096]) == bytes(data[:4096])
        res["seg_%dk" % (seg >> 10)] = {"deflate_e2e_GBps": round(data.size / td / 1e9, 3), "inflate_e2e_GBps": round(data.size / ti / 1e9, 3),
                                       "ratio": round(n.value / data.size, 4), "segments": int(nseg.value)}
    # the reference's own call shape: ONE payload through the batch entry (n = 1).  A member this large is split into primed
    # segments of 64 - 256 KiB, one CTA each (no window reset: the ratio of a single-CTA stream), and decoded as a foreign stream
    ptr1 = (C.c_void_p * 1)(data.ctypes.data); ln1 = (C.c_size_t * 1)(data.size)
    need1 = C.c_size_t(); off1 = (C.c_size_t * 1)(); ol1 = (C.c_size_t * 1)(); ck1 = (C.c_uint32 * 1)(); st1 = (C.c_int * 1)()
    pfn = lambda: L.zipc_b200_deflate_batch(h.ctx.h, 2, 2, 0, 1, ptr1, ln1, cbuf.ctypes.data, cbuf.size, C.byref(need1), off1, ol1, ck1, st1)
    assert pfn() == 0 and st1[0] == 0 and ck1[0] == zlib.crc32(data)
    t0 = time.perf_counter()
    for _ in range(3): pfn()
    tp = (time.perf_counter() - t0) / 3
    plen = int(ol1[0])
    cptr = (C.c_void_p * 1)(cbuf.ctypes.data + int(off1[0])); cln = (C.c_size_t * 1)(plen); mo1 = (C.c_size_t * 1)(data.size)
    need2 = C.c_size_t(); off2 = (C.c_size_t * 1)(); ol2 = (C.c_size_t * 1)(); ck2 = (C.c_uint32 * 1)(); st2 = (C.c_int * 1)()
    qfn = lambda: L.zipc_b200_inflate_batch(h.ctx.h, 2, 0, 1, cptr, cln, mo1, obuf.ctypes.data, obuf.size, C.byref(need2), off2, ol2, ck2, st2)
    assert qfn() == 0 and st2[0] == 0 and ck2[0] == ck1[0]
    t0 = time.perf_counter()
    for _ in range(3): qfn()
    tq = (time.perf_counter() - t0) / 3
    res["one_member_batch_call"] = {"deflate_e2e_GBps": round(data.size / tp / 1e9, 3), "inflate_e2e_GBps": round(data.size / tq / 1e9, 3),
                                    "ratio": round(plen / data.size, 4),
                                    "note": "zipc_b200_deflate_batch / zipc_b200_inflate_batch with n = 1: the member is split into primed segments of 64 - 256 KiB "
                                            "(one CTA each, no ratio loss); the stream is decoded by many warps without an index"}
    # the same data as ONE foreign stream (zlib -6, no index): intra-stream parallel inflate
    zs = zlib.compress(data.tobytes(), 6)[2:-4]
    hz = h.pinned(np.frombuffer(zs, dtype=np.uint8))
    ptr = (C.c_void_p * 1)(hz.ctypes.data)
    ln = (C.c_size_t * 1)(hz.size); mo = (C.c_size_t * 1)(data.size)
    need = C.c_size_t(); off = (C.c_size_t * 1)(); ol = (C.c_size_t * 1)(); ck = (C.c_uint32 * 1)(); stt = (C.c_int * 1)()
    ffn = lambda: L.zipc_b200_inflate_batch(h.ctx.h, 2, 0, 1, ptr, ln, mo, obuf.ctypes.data, obuf.size, C.byref(need), off, ol, ck, stt)
    assert ffn() == 0 and stt[0] == 0 and ck[0] == zlib.crc32(data)
    t0 = time.perf_counter()
    for _ in range(2): ffn()
    tf = (time.perf_counter() - t0) / 2
    res["foreign_zlib6_single_stream"] = {"inflate_e2e_GBps": round(data.size / tf / 1e9, 3), "compressed_bytes": len(zs),
                                          "note": "one RFC 1951 stream made by zlib -6, no index: zipc_b200_inflate_batch with n = 1"}
    return {"workload": "C1: 64 MiB text-v1(seed=1) as one RFC 1951 stream; CRC-32 fused both ways; pinned host buffers in and out", **res}


def run_few_large(h: Harness):
    """The shape of the reference's own benchmark recipe (DEVEL.md:39-52: silesia.zip, 12 members of 5-51 MB, 212 MB): few LARGE
    members instead of many small ones.  Synthetic text of silesia's member sizes; streams made by zlib -6 on the host (a
    foreign encoder, no index); through the plain batch calls with pinned host buffers."""
    from concurrent.futures import ThreadPoolExecutor
    from zipc_b200 import synth
    L = h.L
    sizes = [10192446, 51220480, 9970564, 33553445, 6152192, 10085684, 6627202, 21606400, 7251944, 41458703, 5345280, 8474240]
    datas = [synth.text_v1(700 + i, n) for i, n in enumerate(sizes)]
    with ThreadPoolExecutor(len(sizes)) as ex:
        streams = list(ex.map(lambda d: zlib.compress(d.tobytes(), 6)[2:-4], datas))
    n = len(sizes)
    total = sum(sizes)
    hin = h.pinned(np.concatenate(datas))
    hz = h.pinned(np.frombuffer(b"".join(streams), dtype=np.uint8))
    obuf = h.pinned(np.zeros(total + 64 * n, dtype=np.uint8))
    cbuf = h.pinned(np.zeros(total // 2 + (1 << 20), dtype=np.uint8))
    ptr, ln, mo = (C.c_void_p * n)(), (C.c_size_t * n)(), (C.c_size_t * n)()
    dptr, dln = (C.c_void_p * n)(), (C.c_size_t * n)()
    zo_, do_ = 0, 0
    for i in range(n):
        ptr[i] = hz.ctypes.data + zo_; ln[i] = len(streams[i]); mo[i] = sizes[i]; zo_ += len(streams[i])
        dptr[i] = hin.ctypes.data + do_; dln[i] = sizes[i]; do_ += sizes[i]
    need = C.c_size_t(); off = (C.c_size_t * n)(); ol = (C.c_size_t * n)(); ck = (C.c_uint32 * n)(); st = (C.c_int * n)()
    ifn = lambda: L.zipc_b200_inflate_batch(h.ctx.h, 2, 0, n, ptr, ln, mo, obuf.ctypes.data, obuf.size, C.byref(need), off, ol, ck, st)
    assert ifn() == 0 and all(st[i] == 0 and ck[i] == zlib.crc32(datas[i]) and ol[i] == sizes[i] for i in range(n)), list(st)
    assert bytes(obuf[off[3]:off[3] + 4096]) == bytes(datas[3][:4096])
    t0 = time.perf_counter()
    for _ in range(3): ifn()
    ti = (time.perf_counter() - t0) / 3
    dfn = lambda: L.zipc_b200_deflate_batch(h.ctx.h, 2, 2, 0, n, dptr, dln, cbuf.ctypes.data, cbuf.size, C.byref(need), off, ol, ck, st)
    assert dfn() == 0 and all(st[i] == 0 and ck[i] == zlib.crc32(datas[i]) for i in range(n)), list(st)
    csum = sum(int(ol[i]) for i in range(n))
    assert zlib.decompress(bytes(cbuf[off[4]:off[4] + ol[4]]), -15) == datas[4].tobytes()
    t0 = time.perf_counter()
    for _ in range(3): dfn()
    td = (time.perf_counter() - t0) / 3
    return {"workload": "few large members: 12 members with the sizes of silesia's files (5.3-51.2 MB, %d MB in all), text-v1; pinned host buffers; "
                        "inflate: streams made by zlib -6 on the host, no index; deflate: level default, CRC-32 both ways" % (total // 1000000),
            "members": n, "uncompressed_bytes": total, "inflate_e2e_GBps": round(total / ti / 1e9, 3), "deflate_e2e_GBps": round(total / td / 1e9, 3),
            "zlib6_compressed_bytes": zo_, "deflate_ratio": round(csum / total, 4),
            "note": "every large stream is decoded by many warps (block-start search + speculation), several streams at a time; "
                    "every member is compressed by one CTA per primed segment (64 - 256 KiB, whole waves over the SMs)"}


def run_stream_c5(h: Harness, synth, rank, world, dist, torch, local, slice_bytes=512 << 20, seg=256 << 10):
    """C5: ONE RFC 1951 stream spread over the GPUs of the box (4 GiB at N = 8): every rank compresses its contiguous
    512 MiB slice as a piece of the stream (segment-independent, only the last rank's piece carries BFINAL), the pieces are
    byte aligned so their concatenation in rank order is the stream; back through the per-piece index; the whole-stream
    CRC-32 is the host combine of the slices'.  Pinned host buffers in and out on every rank (end to end); no collective on
    the data path (NCCL only for the max over ranks and the gather of three scalars per rank)."""
    L = h.L
    # every collective below is reached by every rank whatever happens locally: a local failure is a flag, not an exception
    err = None
    try:
        data = h.pinned(make_text(synth, 5 * 64 + rank, slice_bytes))   # (the stream's content: 32 MiB pieces of text-v1, seeds by position)
        cbuf = h.pinned(np.zeros(data.size + (data.size >> 3) + 65536, dtype=np.uint8))
        obuf = h.pinned(np.zeros(data.size, dtype=np.uint8))
        nmax = -(-data.size // seg) + 1
        index = np.zeros((nmax + 1, 2), dtype=np.uint64)
        ip = index.ctypes.data_as(C.POINTER(C.c_uint64))
        n, nseg, crc, crc2, st, olen = C.c_size_t(), C.c_size_t(), C.c_uint32(), C.c_uint32(), C.c_int(), C.c_size_t()
        last_piece = 1 if rank == world - 1 else 0
        dfn = lambda: L.zipc_b200_deflate_segmented(h.ctx.h, 2, data.ctypes.data, data.size, seg, last_piece, cbuf.ctypes.data, cbuf.size,
                                                    C.byref(n), ip, nmax + 1, C.byref(nseg), C.byref(crc))
        ifn = lambda: L.zipc_b200_inflate_segmented(h.ctx.h, cbuf.ctypes.data, n.value, ip, nseg.value, obuf.ctypes.data, obuf.size,
                                                    C.byref(olen), C.byref(crc2), C.byref(st))
        if dfn() != 0 or ifn() != 0:
            err = "segmented call failed: " + L.zipc_b200_last_error(h.ctx.h).decode()
    except Exception as e:
        err = repr(e)
    good = torch.tensor([0.0 if err else 1.0], dtype=torch.float64, device=f"cuda:{local}")
    dist.all_reduce(good, op=dist.ReduceOp.MIN)
    if float(good[0]) == 0.0:
        return {"error": err or "another rank failed"}

    def timed(fn, reps=3):
        torch.cuda.synchronize(); dist.barrier()
        t0 = time.perf_counter()
        for _ in range(reps): fn()
        t = torch.tensor([(time.perf_counter() - t0) / reps], dtype=torch.float64, device=f"cuda:{local}")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t[0])
    td = timed(dfn)
    ti = timed(ifn)
    ok = st.value == 0 and crc2.value == crc.value and olen.value == data.size and bytes(obuf[-4096:]) == bytes(data[-4096:])
    mine = torch.tensor([float(crc.value), float(n.value), 1.0 if ok else 0.0], dtype=torch.float64, device=f"cuda:{local}")
    allv = [torch.zeros_like(mine) for _ in range(world)]
    dist.all_gather(allv, mine)
    whole = int(allv[0][0])
    for k in range(1, world):
        whole = L.zipc_b200_crc32_combine(whole, int(allv[k][0]), data.size)
    total = data.size * world
    return {"workload": "C5: one RFC 1951 stream of %d x 512 MiB text-v1 slices (4 GiB at N = 8), %d KiB segments, default level; pinned host buffers "
                        "in and out on every rank; time = max over ranks" % (world, seg >> 10),
            "total_bytes": total, "deflate_e2e_GBps": round(total / td / 1e9, 2), "inflate_e2e_GBps": round(total / ti / 1e9, 2),
            "ratio": round(sum(float(v[1]) for v in allv) / total, 4), "pieces_ok": int(sum(float(v[2]) for v in allv)), "pieces": world,
            "stream_crc32": "%08x" % whole}


def run_de_yardstick(h: Harness, datas, streams, reps=3):
    """the Blackwell decompression engine on the same members (cuMemBatchDecompressAsync): a yardstick, not a product path"""
    so = os.path.join(ROOT, "tools", "libde_yardstick.so")
    if not os.path.exists(so):
        return {"unsupported": "tools/libde_yardstick.so not built"}
    T = C.CDLL(so)
    n = len(datas)
    keep = [np.ascontiguousarray(s) for s in streams]
    src = (C.c_void_p * n)(*[s.ctypes.data for s in keep])
    exp = (C.c_void_p * n)(*[d.ctypes.data for d in datas])
    sl = np.array([s.size for s in keep], dtype=np.uint64); dl = np.array([d.size for d in datas], dtype=np.uint64)
    ms, nok, msg = C.c_double(), C.c_size_t(), C.create_string_buffer(256)
    T.de_yardstick.argtypes = [C.c_int, C.c_size_t, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.POINTER(C.c_double),
                               C.POINTER(C.c_size_t), C.c_char_p, C.c_size_t]
    rc = T.de_yardstick(h.device, n, src, sl.ctypes.data, exp, dl.ctypes.data, reps, C.byref(ms), C.byref(nok), msg, 256)
    if rc == 1:
        return {"unsupported": msg.value.decode()}
    if rc:
        return {"error": msg.value.decode()}
    U = int(dl.sum())
    return {"de_yardstick_GBps": round(U / (ms.value / 1e3) / 1e9, 2), "ms_per_batch": round(ms.value, 3), "members_ok": int(nok.value), "members": n,
            "note": "cuMemBatchDecompressAsync(CU_MEM_DECOMPRESS_ALGORITHM_DEFLATE), device-resident, same deflate members; no CRC-32"}


def ratio_vs_ref(datas, gpu_sizes, level, sample=160):
    """compressed size of the GPU encoder / compressed size of the reference's encoder (oracle) on the same members, for
    both variants of the reference (SURVEY.md fact 4: code-length frequencies as written / reset per block)"""
    from oracle import zipc_oracle as zo
    idx = list(range(0, len(datas), max(1, len(datas) // sample)))[:sample]
    ours = int(sum(int(gpu_sizes[i]) for i in idx)); U = int(sum(datas[i].size for i in idx))
    out = {"sample_members": len(idx), "ratio_gpu": round(ours / U, 4)}
    cores = os.cpu_count() or 1
    for name, keep in (("as_written", True), ("freqs_reset", False)):
        zo.set_keep_codelen_freqs(keep)
        with ThreadPoolExecutor(max_workers=cores) as ex:
            ref = sum(ex.map(lambda i: len(zo.deflate(datas[i].tobytes(), level)), idx))
        out["ratio_ref_" + name] = round(ref / U, 4)
        out["ratio_vs_ref_" + name] = round(ours / ref, 4)
    zo.set_keep_codelen_freqs(True)
    return out


# ---------------------------------------------------------------------------------------------------
# CPU side: the reference's algorithm (oracle = C restatement; kind "port") on the host cores
# ---------------------------------------------------------------------------------------------------
def cpu_crc32(host: np.ndarray, budget_s=8.0):
    from oracle import zipc_oracle as zo
    L = zo.lib()
    n = host.size
    t0 = time.perf_counter()
    reps = 0
    while True:
        L.zo_crc32(C.cast(host.ctypes.data, C.c_char_p), n)
        reps += 1
        if time.perf_counter() - t0 > budget_s or reps >= 8:
            break
    dt = time.perf_counter() - t0
    t1 = time.perf_counter(); zlib.crc32(host[: 256 << 20]); tz = time.perf_counter() - t1   # a familiar yardstick (SURVEY.md 8d)
    return {"value": round(n * reps / dt / 1e9, 3), "unit": "GB/s", "cores": 1, "kind": "port",
            "sample": f"{reps} x full 1 GiB buffer, Crc_32.string restated in C (oracle/zipc_oracle.c), 1 thread: the reference hashes one string on one core",
            "zlib_crc32_yardstick_GBps": round((256 << 20) / tz / 1e9, 3)}


def cpu_codec(which, datas, streams=None, level="default", budget_s=10.0, all_members=False):
    """one member per thread from a shared queue over all host cores (the reference's natural multi-core use).
    Returns (baseline dict, list of compressed streams of the sample when deflating)."""
    from oracle import zipc_oracle as zo
    zo.lib()
    cores = os.cpu_count() or 1
    n = len(datas)

    def work(i):
        if which == "inflate":
            zo.inflate_and_crc_32(bytes(streams[i]), datas[i].size)
            return None
        return zo.crc_32_and_deflate(datas[i].tobytes(), level)[1]
    if all_members:
        sample = list(range(n))
    else:  # bounded sample: as many members as fit the budget, estimated from a probe
        probe = list(range(min(n, cores)))
        t0 = time.perf_counter()
        with ThreadPoolExecutor(max_workers=cores) as ex:
            list(ex.map(work, probe))
        rate = sum(datas[i].size for i in probe) / max(time.perf_counter() - t0, 1e-6)
        target, sample, acc = rate * budget_s, [], 0
        for i in range(n):
            if acc >= target:
                break
            sample.append(i); acc += datas[i].size
    t0 = time.perf_counter()
    with ThreadPoolExecutor(max_workers=cores) as ex:
        outs = list(ex.map(work, sample))
    dt = time.perf_counter() - t0
    done = sum(datas[i].size for i in sample)
    fn = "inflate_and_crc_32" if which == "inflate" else "crc_32_and_deflate level " + level
    return {"value": round(done / dt / 1e9, 4), "unit": "GB/s", "cores": cores, "kind": "port",
            "sample": f"{len(sample)} of {n} members ({done/1e6:.0f} MB uncompressed), one member per thread over {cores} threads, {fn} restated in C (oracle/)"}, outs


def reference_arm(args):
    """--impl reference: the reference's CPU implementation of the path on this box's host cores (never loads the GPU library)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import synth                      # same generators, own shared object
    from oracle import zipc_oracle as zo
    which, steps, warmup = args.workload, args.steps, args.warmup
    cores = os.cpu_count() or 1
    if which == "crc32":
        # weak scaling: N GPUs hash N independent 1 GiB buffers, so the reference hashes N buffers too, one string per core
        nbuf = max(1, min(args.gpus, cores))
        hosts = [synth.rand_v1(2 + r, GiB) for r in range(nbuf)]
        L = zo.lib()
        one = lambda hbuf: L.zo_crc32(C.cast(hbuf.ctypes.data, C.c_char_p), hbuf.size)

        def step():
            with ThreadPoolExecutor(max_workers=nbuf) as ex:
                list(ex.map(one, hosts))
            return GiB * nbuf
        used = nbuf
        sample = f"each step = Crc_32.string (C restatement) over {nbuf} x 1 GiB buffer(s), one string per thread (one string = one core in the reference)"
    else:
        datas = make_members(synth, args.members, 1000)
        zo.lib()
        if which == "inflate":
            with ThreadPoolExecutor(max_workers=cores) as ex:
                streams = list(ex.map(lambda d: zo.deflate(d.tobytes(), args.level), datas))
            work = lambda i: (zo.inflate_and_crc_32(streams[i], datas[i].size), datas[i].size)[1]
        else:
            work = lambda i: (zo.crc_32_and_deflate(datas[i].tobytes(), args.level), datas[i].size)[1]
        # a step is a bounded sample of the 10k members, sized from a probe to about one second of all cores
        probe = list(range(min(len(datas), 2 * cores)))
        t0 = time.perf_counter()
        with ThreadPoolExecutor(max_workers=cores) as ex:
            done = sum(ex.map(work, probe))
        rate = done / max(time.perf_counter() - t0, 1e-6)
        target, idx, acc = rate * 1.0, [], 0
        for i in range(len(datas)):
            if acc >= target and len(idx) >= cores:
                break
            idx.append(i); acc += datas[i].size

        def step():
            with ThreadPoolExecutor(max_workers=cores) as ex:
                return sum(ex.map(work, idx))
        used = cores
        fn = "inflate_and_crc_32" if which == "inflate" else "crc_32_and_deflate"
        sample = (f"each step = the first {len(idx)} of the {len(datas)} members ({acc/1e6:.0f} MB uncompressed; a rate, so the sample does not "
                  f"change the metric), {fn} level {args.level} restated in C (oracle/), one member per thread over {cores} threads")
    for _ in range(min(warmup, 2)):
        step()
    t0 = time.perf_counter()
    done = 0
    for _ in range(steps):
        done += step()
    dt = time.perf_counter() - t0
    value = done / dt / 1e9
    line = {"impl": "reference", "metric": METRIC[which], "value": round(value, 4), "unit": "GB/s", "n_gpus": args.gpus, "steps": steps,
            "warmup": warmup, "ms_per_step": round(dt / steps * 1e3, 3), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": make_config(which, args.level, args.members),
            "note": "the reference is OCaml (no toolchain in this image): timed through its C restatement oracle/zipc_oracle.c",
            "cpu_baseline": {"value": round(value, 4), "unit": "GB/s", "cores": used, "kind": "port", "sample": sample},
            "e2e": {"value": round(value, 4), "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))
    return 0


# ---------------------------------------------------------------------------------------------------
def strong_scaling(world, datas, streams, host_crc_buf, single):
    """Rank 0 only: ONE member set / ONE buffer over all `world` GPUs through the box-wide entry points, pinned host buffers,
    gather + CRC combine inside the timed region.  `single` holds the one-GPU e2e seconds of the same calls."""
    from zipc_b200 import zipc_deflate as zd
    m = zd.MultiContext((1 << world) - 1)
    L = m.L
    out = {"devices": m.devices, "entry_points": "zipc_b200_multi_deflate_batch / zipc_b200_multi_inflate_batch / zipc_b200_multi_crc32"}
    try:
        n = len(datas)
        U = int(sum(d.size for d in datas))

        def pin(a):
            p = C.c_void_p()
            assert L.zipc_b200_host_alloc(max(a.size, 1), C.byref(p)) == 0
            o = np.ctypeslib.as_array((C.c_uint8 * max(a.size, 1)).from_address(p.value))[:a.size]
            o[:] = a
            return o, p
        pins = []
        src, p = pin(np.concatenate(datas)); pins.append(p)
        soff = np.concatenate([[0], np.cumsum([d.size for d in datas])[:-1]]).astype(np.uint64)
        slen = np.array([d.size for d in datas], dtype=np.uint64)
        ptrs = (C.c_void_p * n)(*[src.ctypes.data + int(o) for o in soff])
        arena, p = pin(np.zeros(U + 16 * n + 4096, dtype=np.uint8)); pins.append(p)
        need = C.c_size_t(); off = np.zeros(n, dtype=np.uint64); dl = np.zeros(n, dtype=np.uint64)
        ck = np.zeros(n, dtype=np.uint32); st = np.zeros(n, dtype=np.int32)

        def dfn():
            rc = L.zipc_b200_multi_deflate_batch(m.h, 2, 2, 0, n, ptrs, P(slen, C.c_size_t), arena.ctypes.data, arena.size, C.byref(need),
                                                 P(off, C.c_size_t), P(dl, C.c_size_t), P(ck, C.c_uint32), P(st, C.c_int))
            assert rc == 0 and (st == 0).all(), rc
        dfn()
        t0 = time.perf_counter(); dfn(); dfn(); td = (time.perf_counter() - t0) / 2
        k = n // 2
        assert zlib.decompress(arena[int(off[k]):int(off[k]) + int(dl[k])].tobytes(), -15) == datas[k].tobytes() and int(ck[k]) == zlib.crc32(datas[k])
        out["deflate"] = {"e2e_GBps": round(U / td / 1e9, 3), "speedup_vs_1gpu_e2e": round(single["deflate"] / td, 3) if single.get("deflate") else None}
        # inflate of the same set
        cs, p = pin(np.concatenate([np.asarray(s) for s in streams])); pins.append(p)
        coff = np.concatenate([[0], np.cumsum([len(s) for s in streams])[:-1]]).astype(np.uint64)
        clen = np.array([len(s) for s in streams], dtype=np.uint64)
        cptrs = (C.c_void_p * n)(*[cs.ctypes.data + int(o) for o in coff])

        def ifn():
            rc = L.zipc_b200_multi_inflate_batch(m.h, 2, 0, n, cptrs, P(clen, C.c_size_t), P(slen, C.c_size_t), arena.ctypes.data, arena.size,
                                                 C.byref(need), P(off, C.c_size_t), P(dl, C.c_size_t), P(ck, C.c_uint32), P(st, C.c_int))
            assert rc == 0 and (st == 0).all() and (dl == slen).all(), rc
        ifn()
        t0 = time.perf_counter(); ifn(); ifn(); ti = (time.perf_counter() - t0) / 2
        assert arena[int(off[k]):int(off[k]) + int(dl[k])].tobytes() == datas[k].tobytes()
        out["inflate"] = {"e2e_GBps": round(U / ti / 1e9, 3), "speedup_vs_1gpu_e2e": round(single["inflate"] / ti, 3) if single.get("inflate") else None}
        # one 1 GiB buffer: slices + host combine
        if host_crc_buf is not None:
            o = C.c_uint32()
            cfn = lambda: L.zipc_b200_multi_crc32(m.h, host_crc_buf.ctypes.data, host_crc_buf.size, C.byref(o))
            assert cfn() == 0
            t0 = time.perf_counter(); cfn(); cfn(); cfn(); tcr = (time.perf_counter() - t0) / 3
            assert o.value == zlib.crc32(host_crc_buf)
            out["crc32"] = {"e2e_GBps": round(host_crc_buf.size / tcr / 1e9, 2), "speedup_vs_1gpu_e2e": round(single["crc32"] / tcr, 3) if single.get("crc32") else None,
                            "note": "one buffer cut into N slices, N-1 zipc_b200_crc32_combine steps on the host"}
        out["note"] = ("strong scaling: total work fixed, one host process drives all GPUs; bounded by the host side of the PCIe copies "
                       "(all GPUs of this box hang off one host memory system)")
        for p in pins:
            L.zipc_b200_host_free(p)
    finally:
        m.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", choices=["crc32", "inflate", "deflate"], default="deflate")
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--no-also", action="store_true", help="skip the secondary workloads")
    ap.add_argument("--members", type=int, default=10000)
    ap.add_argument("--level", choices=["fast", "default", "best"], default="default", help="deflate level of the codec workloads")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the headline call returned in its last timed step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps is None:
        args.steps = 20 if args.workload == "crc32" else 5
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of this project's GPU path: it does not apply to --impl reference")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        return reference_arm(args)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # the library pipelines a large batch in groups, one host thread each; it sizes that by the cores per VISIBLE GPU, but under
    # torchrun every rank sees all GPUs of the box while `world` ranks share its cores: tell it this process's share
    os.environ.setdefault("ZIPC_B200_PIPE", str(max(4, min(24, 2 * (os.cpu_count() or 8) // max(1, world)))))
    import torch
    dist, cpu_group = None, None
    if world > 1:
        import torch.distributed as dist
        torch.cuda.set_device(local)
        dist.init_process_group(backend="nccl", device_id=torch.device(f"cuda:{local}"))
        cpu_group = dist.new_group(backend="gloo")
    from zipc_b200 import synth
    numa = bind_near_gpu(local) if world > 1 else None   # before any pinned allocation: first touch decides where the pages live
    h = Harness(local)
    peak, peak_src = measured_peak_gbs()

    def barrier():
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    def reduce(r):
        """max over ranks of the device time and of the end-to-end time; units summed over ranks"""
        vals = torch.tensor([r["total_ms"], r["e2e_s"] or 0.0], dtype=torch.float64, device=f"cuda:{local}")
        units = torch.tensor([float(r["units"])], dtype=torch.float64, device=f"cuda:{local}")
        if dist is not None:
            dist.all_reduce(vals, op=dist.ReduceOp.MAX)
            dist.all_reduce(units, op=dist.ReduceOp.SUM)
        r["value"] = float(units[0]) * r["steps"] / (float(vals[0]) / 1e3) / 1e9
        r["e2e"] = float(units[0]) / float(vals[1]) / 1e9 if float(vals[1]) > 0 else None
        r["ms_per_step"] = float(vals[0]) / r["steps"]
        return r

    def measured(fn):
        barrier()
        with ClockSampler(local) as cs:
            r = fn()
        barrier()
        r["clocks"] = cs.summary()
        return reduce(r)

    def roofline(r):
        if not r.get("kernel_ms"):
            return None
        ach = r["algo_bytes"] / (r["kernel_ms"] / 1e3) / 1e9
        which = {"crc32_tiles_kernel": "crc32", "inflate_kernel<false>": "inflate", "deflate_kernel": "deflate"}.get(r["kernel"])
        return {"bound": "hbm", "achieved": round(ach, 1), "peak": peak, "unit": "GB/s", "frac": round(ach / peak, 4),
                "traffic": ncu_traffic(which) if which else None,
                "kernel": r["kernel"], "kernel_ms": round(r["kernel_ms"], 4), "algorithmic_bytes": int(r["algo_bytes"]), "peak_source": peak_src,
                "ncu": {k: v for k, v in ncu_capture(which).items() if k not in ("traffic_bytes", "kernel")} if which else None}

    def brief(r, which, level=None):
        d = {"metric": METRIC[which], "value": round(r["value"], 2), "unit": "GB/s", "e2e": round(r["e2e"], 3) if r.get("e2e") else None,
             "kernel_ms": round(r["kernel_ms"], 4) if r.get("kernel_ms") else None, "roofline": roofline(r),
             "workload": workload_desc(which, level or args.level, args.members), **r["extra"]}
        return d

    which = args.workload
    datas = make_members(synth, args.members, 1000 + rank * args.members) if (which != "crc32" or not args.no_also) else None
    streams = None
    single_e2e = {}
    also = {}

    def get_streams():
        nonlocal streams
        if streams is None:
            res = h.ctx.deflate_batch(datas, args.level, 2)
            assert all(x[0] == 0 for x in res)
            streams = [x[1] for x in res]
        return streams

    # ---- headline ---------------------------------------------------------------------------------------------------
    dump = bool(args.dump_outputs) and rank == 0
    if which == "deflate":
        r = measured(lambda: run_deflate(h, datas, args.level, args.steps, args.warmup, keep_streams=True, dump=dump))
        streams = r.pop("streams", None)
        single_e2e["deflate"] = r["e2e_s"]
    elif which == "inflate":
        get_streams()
        r = measured(lambda: run_inflate(h, datas, streams, args.steps, args.warmup, dump=dump))
        single_e2e["inflate"] = r["e2e_s"]
    else:
        r = measured(lambda: run_crc32(h, args.steps, args.warmup, rank, dump=dump))
        single_e2e["crc32"] = r["e2e_s"]
    outputs = r.pop("outputs")
    if dump:
        write_outputs(args.dump_outputs, outputs)
    line = {"metric": METRIC[which], "value": round(r["value"], 2), "unit": "GB/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": round(r["ms_per_step"], 4), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": make_config(which, args.level, args.members),
            "detail": {"per_gpu_bytes": int(r["units"]), **r["extra"]},
            "clocks": r["clocks"],
            "e2e": {"value": round(r["e2e"], 3), "unit": "GB/s", "h2d_bytes_per_step": int(r["h2d"]), "d2h_bytes_per_step": int(r["d2h"]),
                    "note": "C-ABI call with pinned host buffers (codec members lie in one pinned buffer, like an in-memory archive); H2D + kernels + D2H per step"},
            "gpu_launches": int(r["launches"]), "roofline": roofline(r)}
    if numa:
        line["detail"]["host_cpus_per_rank"] = numa   # (ranks are bound to the CPUs local to their GPU)
    head_sizes = r.get("sizes")
    crc_host = r.get("host")
    oracle_streams = None
    if rank == 0:
        try:
            if which == "deflate":
                line["ratio_vs_ref"] = ratio_vs_ref(datas, head_sizes, args.level)
            if world == 1:
                if which == "crc32":
                    line["cpu_baseline"] = cpu_crc32(crc_host)
                elif which == "deflate" and not args.no_also and args.level == "default":
                    # the full member set through the reference's encoder: it is also the oracle-made C3 archive's payloads
                    line["cpu_baseline"], oracle_streams = cpu_codec("deflate", datas, level=args.level, all_members=True)
                else:
                    line["cpu_baseline"], _ = cpu_codec(which, datas, get_streams() if which == "inflate" else None, args.level)
        except Exception as e:
            line["cpu_baseline_error"] = repr(e)

    # ---- the rest of the metric, at every N ----------------------------------------------------------------------------
    if not args.no_also:
        def guard(name, fn):
            try:
                also[name] = fn()
            except Exception as e:  # never lose the headline line to a secondary workload
                also[name] = {"error": repr(e)}
            h.free_pins()

        def lvl_entry(level):
            rr = measured(lambda: run_deflate(h, datas, level, 2, 3, e2e=False))
            d = brief(rr, "deflate", level)
            if rank == 0:
                d["ratio_vs_ref"] = ratio_vs_ref(datas, rr["sizes"], level, sample=64 if level == "best" else 160)
            return d
        if which != "deflate":
            guard("deflate_" + args.level, lambda: lvl_entry(args.level))
        for level in ("fast", "default", "best"):
            if level != args.level:
                guard("deflate_" + level, lambda level=level: lvl_entry(level))

        def none_entry():  # level `None: stored blocks, byte-identical to the reference's output -- a copy with block headers
            rr = measured(lambda: run_deflate(h, datas, "none", 3, 3, e2e=False))
            rr["kernel"] = "stored_kernel"
            rr["algo_bytes"] = 2 * rr["units"]   # every input byte read once and written once (+ 5 bytes per 65,534)
            d = brief(rr, "deflate", "none")
            d["note"] = "stored blocks of 65,534 bytes (zipc_deflate.ml:747-750, 1106-1116); roofline: bytes read + bytes written over the kernel's time"
            return d
        guard("deflate_none", none_entry)
        if which != "inflate":
            def inflate_entry():
                get_streams()
                rr = measured(lambda: run_inflate(h, datas, streams, 3, 3))
                single_e2e["inflate"] = rr["e2e_s"]
                d = brief(rr, "inflate")
                d["streams"] = "made by the GPU encoder (level %s)" % args.level
                if rank == 0 and world == 1:
                    d["cpu_baseline"], _ = cpu_codec("inflate", datas, streams, budget_s=6.0)
                return d
            guard("inflate", inflate_entry)
        if which != "crc32":
            def crc_entry():
                nonlocal crc_host
                rr = measured(lambda: run_crc32(h, 10, 3, rank))
                single_e2e["crc32"] = rr["e2e_s"]
                crc_host = rr["host"]
                d = brief(rr, "crc32")
                if rank == 0 and world == 1:
                    d["cpu_baseline"] = cpu_crc32(crc_host, budget_s=4.0)
                return d
            guard("crc32", crc_entry)
        if world == 1:
            def foreign():
                def comp(d):
                    c = zlib.compressobj(6, zlib.DEFLATED, -15)
                    return np.frombuffer(c.compress(d.tobytes()) + c.flush(), dtype=np.uint8)
                with ThreadPoolExecutor(max_workers=os.cpu_count() or 4) as ex:
                    zs = list(ex.map(comp, datas))
                rr = measured(lambda: run_inflate(h, datas, zs, 3, 3, e2e=False))
                d = brief(rr, "inflate")
                d["streams"] = "made by zlib -6 on the host (foreign encoder: longer matches, ~16k-symbol blocks)"
                return d
            guard("inflate_zlib6_streams", foreign)
            if oracle_streams is not None:
                def oracle_made():
                    os_ = [np.frombuffer(s, dtype=np.uint8) for s in oracle_streams]
                    rr = measured(lambda: run_inflate(h, datas, os_, 3, 3, e2e=True))
                    d = brief(rr, "inflate")
                    d["streams"] = "made by the oracle (the reference's encoder restated, level default, as written): SURVEY.md 8d's C3 archive"
                    return d
                guard("inflate_oracle_streams", oracle_made)

                def archive():
                    from oracle import zipc_oracle as zo
                    ms = [zo.member_make(b"m/%05d.txt" % i, compression=8, compressed_bytes=oracle_streams[i], decompressed_size=datas[i].size,
                                         crc32=zlib.crc32(datas[i])) for i in range(len(datas))]
                    return run_archive(h, datas, zo.zip_encode(ms))
                guard("archive", archive)
            else:
                guard("archive", lambda: run_archive(h, datas))
            guard("stream_c1", lambda: run_stream_c1(h))
            guard("few_large_members", lambda: run_few_large(h))
            guard("de_yardstick", lambda: run_de_yardstick(h, datas, get_streams()))
        else:
            # C5: one stream over all GPUs of the box (every rank takes part)
            def c5():
                d = run_stream_c5(h, synth, rank, world, dist, torch, local)
                return d
            guard("stream_c5", c5)
            # strong scaling: rank 0 drives all GPUs through the box-wide entry points; the other ranks stay off their GPUs
            get_streams()
            torch.cuda.synchronize()
            dist.barrier(group=cpu_group)
            if rank == 0:
                guard("strong_scaling", lambda: strong_scaling(world, datas, streams, crc_host, single_e2e))
            dist.barrier(group=cpu_group)
        line["also"] = also
    if rank == 0:
        print(json.dumps(line))
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
