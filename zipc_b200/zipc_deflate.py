"""Host-side mirror of the reference's `Zipc_deflate` module over the C ABI of libzipc_b200.so.

Same names, argument meaning and error behaviour as /root/reference/src/zipc_deflate.mli, so the
parity tests read like the reference's own tests (test/test.ml):

    Crc_32.string / Adler_32.string                       zipc_deflate.mli:24-75
    inflate / inflate_and_crc_32 / inflate_and_adler_32    zipc_deflate.mli:79-102
    zlib_decompress                                        zipc_deflate.mli:104-118
    deflate / crc_32_and_deflate / adler_32_and_deflate    zipc_deflate.mli:128-149
    zlib_compress                                          zipc_deflate.mli:151-162

OCaml's `('a, string) result` becomes Ok(value) / Error(message).  Every function has a `_batch`
form taking a list of inputs: one call per ZIP member cannot feed a GPU (SURVEY.md 8b).

All compute happens in the CUDA library; this file only marshals buffers.  (The OCaml binding with
the same shape is ocaml/zipc_cuda.ml; see INTEGRATION.md.)
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Iterable, Sequence

import numpy as np

from . import _lib
from ._lib import (ADLER_REF_COMPAT, ADLER_RFC1950, CK_ADLER32, CK_CRC32, CK_NONE, SIZE_UNKNOWN)

LEVELS = {"none": 0, "fast": 1, "default": 2, "best": 3}


# ---- ('a, string) result -------------------------------------------------------------------------
class Ok:
    __slots__ = ("value",)

    def __init__(self, value):
        self.value = value

    def is_ok(self):
        return True

    def is_error(self):
        return False

    def get_ok(self):
        return self.value

    def __repr__(self):
        return f"Ok({self.value!r})"


class Error:
    __slots__ = ("message", "status", "info")

    def __init__(self, message, status=0, info=None):
        self.message, self.status, self.info = message, status, info

    def is_ok(self):
        return False

    def is_error(self):
        return True

    def get_ok(self):
        raise ValueError(f"Result.get_ok on Error {self.message!r}")

    def __repr__(self):
        return f"Error({self.message!r})"


class ZipcB200Error(RuntimeError):
    """Call-level failure (CUDA, memory, arguments): no analogue in the reference."""


def strerror(status: int) -> str:
    return _lib.lib().zipc_b200_strerror(status).decode()


def _crc_error(expect: int, found: int) -> str:
    # "Checksum mismatch, expected %lx found %lx)" -- zipc_deflate.ml:103-104, stray ')' included
    return "Checksum mismatch, expected %x found %x)" % (expect, found)


def _as_view(b) -> np.ndarray:
    """Zero-copy uint8 view of bytes / bytearray / memoryview / ndarray."""
    if isinstance(b, np.ndarray):
        return b.reshape(-1).view(np.uint8)
    return np.frombuffer(b, dtype=np.uint8)


def _slice(s, start, length):
    v = _as_view(s)
    n = v.size
    if length is None:
        length = n - start
    if start < 0 or length < 0 or start + length > n:
        raise ValueError("index out of bounds")  # OCaml: Invalid_argument
    return v[start:start + length]


class Context:
    """One zipc_b200_ctx: a CUDA device, a stream and the library's grow-only work buffers."""

    def __init__(self, device: int | None = None):
        self.L = _lib.lib()
        if device is None:
            device = int(os.environ.get("ZIPC_B200_DEVICE", os.environ.get("LOCAL_RANK", "0")))
        h = C.c_void_p()
        st = self.L.zipc_b200_ctx_create(device, C.byref(h))
        if st:
            raise ZipcB200Error(f"zipc_b200_ctx_create(device={device}): {strerror(st)} -- libzipc_b200 has no CPU fallback")
        self.h, self.device = h, device

    def close(self):
        if getattr(self, "h", None):
            self.L.zipc_b200_ctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- helpers
    def _check(self, st, what):
        if st:
            raise ZipcB200Error(f"{what}: {strerror(st)} [{self.L.zipc_b200_last_error(self.h).decode()}]")

    @property
    def launches(self) -> int:
        return self.L.zipc_b200_ctx_launches(self.h)

    @property
    def stream(self) -> int:
        return self.L.zipc_b200_ctx_stream(self.h) or 0

    @property
    def parallel_streams(self) -> tuple[int, int]:
        """(large streams inflated in parallel inside the stream, large streams handed back to the one-warp decoder)"""
        return self.L.zipc_b200_ctx_counter(self.h, 1), self.L.zipc_b200_ctx_counter(self.h, 2)

    @property
    def parallel_counters(self) -> tuple[int, int, int, int]:
        """parallel_streams, then the many-warp decoder's speculation passes (none for a plan kept from the sizing pass of the
        same call) and the chunks it resolved"""
        return tuple(self.L.zipc_b200_ctx_counter(self.h, k) for k in (1, 2, 3, 4))

    @staticmethod
    def _ptr_arrays(items: Sequence[np.ndarray]):
        n = len(items)
        ptrs = (C.c_void_p * max(n, 1))()
        lens = (C.c_size_t * max(n, 1))()
        for i, v in enumerate(items):
            ptrs[i] = v.ctypes.data if v.size else None
            lens[i] = v.size
        return ptrs, lens

    # -- checksums
    def crc32(self, s) -> int:
        v = _as_view(s)
        out = C.c_uint32()
        self._check(self.L.zipc_b200_crc32(self.h, v.ctypes.data if v.size else None, v.size, C.byref(out)), "crc32")
        return out.value

    def adler32(self, s, mode: int = ADLER_REF_COMPAT) -> int:
        v = _as_view(s)
        out = C.c_uint32()
        self._check(self.L.zipc_b200_adler32(self.h, v.ctypes.data if v.size else None, v.size, mode, C.byref(out)), "adler32")
        return out.value

    def crc32_batch(self, items: Iterable) -> list[int]:
        vs = [_as_view(x) for x in items]
        ptrs, lens = self._ptr_arrays(vs)
        out = (C.c_uint32 * max(len(vs), 1))()
        self._check(self.L.zipc_b200_crc32_batch(self.h, len(vs), ptrs, lens, out), "crc32_batch")
        return list(out[:len(vs)])

    # -- codecs: shared driver for the four batch entry points with an output arena
    def _arena_call(self, call, n):
        """call(dst, cap, need, off, len) -> status.  Runs once without an arena, then fetches."""
        need = C.c_size_t()
        off = (C.c_size_t * max(n, 1))()
        ln = (C.c_size_t * max(n, 1))()
        st = call(None, 0, C.byref(need), off, ln)
        if st not in (_lib.OK, _lib.ERR_DST_TOO_SMALL):
            self._check(st, "batch call")
        arena = np.empty(max(need.value, 1), dtype=np.uint8)
        if st == _lib.ERR_DST_TOO_SMALL:
            self._check(self.L.zipc_b200_fetch(self.h, arena.ctypes.data, arena.size), "fetch")
        return arena, off, ln

    def inflate_batch(self, items: Sequence, decompressed_sizes: Sequence[int | None] | None = None,
                      crc_op: int = CK_NONE, adler_mode: int = ADLER_REF_COMPAT):
        """-> list of (status, bytes-like output, checksum)."""
        vs = [_as_view(x) for x in items]
        n = len(vs)
        ptrs, lens = self._ptr_arrays(vs)
        mo = (C.c_size_t * max(n, 1))()
        for i in range(n):
            d = None if decompressed_sizes is None else decompressed_sizes[i]
            mo[i] = SIZE_UNKNOWN if d is None else d
        ck = (C.c_uint32 * max(n, 1))()
        stt = (C.c_int * max(n, 1))()
        arena, off, ln = self._arena_call(
            lambda dst, cap, need, o, l: self.L.zipc_b200_inflate_batch(self.h, crc_op, adler_mode, n, ptrs, lens, mo,
                                                                        dst, cap, need, o, l, ck, stt), n)
        return [(stt[i], arena[off[i]:off[i] + ln[i]], ck[i]) for i in range(n)]

    def zlib_decompress_batch(self, items: Sequence, decompressed_sizes=None, adler_mode: int = ADLER_REF_COMPAT):
        """-> list of (status, output, expect, found)."""
        vs = [_as_view(x) for x in items]
        n = len(vs)
        ptrs, lens = self._ptr_arrays(vs)
        mo = (C.c_size_t * max(n, 1))()
        for i in range(n):
            d = None if decompressed_sizes is None else decompressed_sizes[i]
            mo[i] = SIZE_UNKNOWN if d is None else d
        ex, fo = (C.c_uint32 * max(n, 1))(), (C.c_uint32 * max(n, 1))()
        stt = (C.c_int * max(n, 1))()
        arena, off, ln = self._arena_call(
            lambda dst, cap, need, o, l: self.L.zipc_b200_zlib_decompress_batch(self.h, adler_mode, n, ptrs, lens, mo, dst,
                                                                                cap, need, o, l, ex, fo, stt), n)
        return [(stt[i], arena[off[i]:off[i] + ln[i]], ex[i], fo[i]) for i in range(n)]

    def deflate_batch(self, items: Sequence, level: str = "default", crc_op: int = CK_NONE,
                      adler_mode: int = ADLER_REF_COMPAT):
        """-> list of (status, compressed bytes-like, checksum of the input)."""
        vs = [_as_view(x) for x in items]
        n = len(vs)
        ptrs, lens = self._ptr_arrays(vs)
        ck = (C.c_uint32 * max(n, 1))()
        stt = (C.c_int * max(n, 1))()
        lv = LEVELS[level]
        arena, off, ln = self._arena_call(
            lambda dst, cap, need, o, l: self.L.zipc_b200_deflate_batch(self.h, lv, crc_op, adler_mode, n, ptrs, lens, dst,
                                                                        cap, need, o, l, ck, stt), n)
        return [(stt[i], arena[off[i]:off[i] + ln[i]], ck[i]) for i in range(n)]

    def zlib_compress_batch(self, items: Sequence, level: str = "default", adler_mode: int = ADLER_REF_COMPAT):
        vs = [_as_view(x) for x in items]
        n = len(vs)
        ptrs, lens = self._ptr_arrays(vs)
        ad = (C.c_uint32 * max(n, 1))()
        stt = (C.c_int * max(n, 1))()
        lv = LEVELS[level]
        arena, off, ln = self._arena_call(
            lambda dst, cap, need, o, l: self.L.zipc_b200_zlib_compress_batch(self.h, lv, adler_mode, n, ptrs, lens, dst, cap,
                                                                              need, o, l, ad, stt), n)
        return [(stt[i], arena[off[i]:off[i] + ln[i]], ad[i]) for i in range(n)]


    # -- one large stream as independent segments (configs 1 and 5)
    def deflate_segmented(self, s, level: str = "default", segment_size: int = 256 << 10, last_piece: bool = True, primed: bool = False):
        """-> (stream bytes-like, index ndarray[(nseg+1), 2] of (compressed, uncompressed) offsets, crc32 of s).
        primed: every segment sees the 32 KiB of input before it (zipc_b200_deflate_primed): no ratio loss, but the stream
        is then decoded like a foreign one (inflate_batch), not by inflate_segmented."""
        v = _as_view(s)
        nseg_max = max(1, -(-v.size // segment_size))
        index = np.zeros((nseg_max + 1, 2), dtype=np.uint64)
        n, nseg, crc = C.c_size_t(), C.c_size_t(), C.c_uint32()
        args = (self.h, LEVELS[level], v.ctypes.data if v.size else None, v.size, segment_size, int(last_piece))
        fn = self.L.zipc_b200_deflate_primed if primed else self.L.zipc_b200_deflate_segmented
        st = fn(*args, None, 0, C.byref(n), index.ctypes.data_as(C.POINTER(C.c_uint64)), nseg_max + 1, C.byref(nseg), C.byref(crc))
        if st != _lib.ERR_DST_TOO_SMALL:
            self._check(st, "deflate_segmented")
        out = np.empty(max(n.value, 1), dtype=np.uint8)
        self._check(self.L.zipc_b200_fetch(self.h, out.ctypes.data, out.size), "fetch")
        return out[:n.value], index[:nseg.value + 1], crc.value

    def inflate_segmented(self, stream, index):
        """-> (status, output bytes-like, crc32 of the output)"""
        v = _as_view(stream)
        index = np.ascontiguousarray(index, dtype=np.uint64)
        nseg = index.shape[0] - 1
        out = np.empty(max(int(index[nseg, 1]), 1), dtype=np.uint8)
        n, crc, st = C.c_size_t(), C.c_uint32(), C.c_int()
        rc = self.L.zipc_b200_inflate_segmented(self.h, v.ctypes.data if v.size else None, v.size,
                                                index.ctypes.data_as(C.POINTER(C.c_uint64)), nseg, out.ctypes.data, out.size,
                                                C.byref(n), C.byref(crc), C.byref(st))
        self._check(rc, "inflate_segmented")
        return st.value, out[:n.value], crc.value


class MultiContext:
    """zipc_b200_mctx: one call drives every selected GPU of the node (device_mask bit d = CUDA device d; 0 = all).
    Members of a batch are partitioned over the devices inside the library; results come back in input order."""

    def __init__(self, device_mask: int = 0):
        self.L = _lib.lib()
        h = C.c_void_p()
        st = self.L.zipc_b200_mctx_create(device_mask, C.byref(h))
        if st:
            raise ZipcB200Error(f"zipc_b200_mctx_create(mask={device_mask:#x}): {strerror(st)} -- libzipc_b200 has no CPU fallback")
        self.h = h
        self.devices = self.L.zipc_b200_mctx_device_count(h)

    def close(self):
        if getattr(self, "h", None):
            self.L.zipc_b200_mctx_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _check(self, st, what):
        if st:
            raise ZipcB200Error(f"{what}: {strerror(st)} [{self.L.zipc_b200_mctx_last_error(self.h).decode()}]")

    @property
    def launches(self) -> int:
        return sum(self.L.zipc_b200_ctx_launches(self.L.zipc_b200_mctx_ctx(self.h, k)) for k in range(self.devices))

    def crc32(self, s) -> int:
        v = _as_view(s)
        out = C.c_uint32()
        self._check(self.L.zipc_b200_multi_crc32(self.h, v.ctypes.data if v.size else None, v.size, C.byref(out)), "multi_crc32")
        return out.value

    def _arena_call(self, call, n):
        need = C.c_size_t()
        off = (C.c_size_t * max(n, 1))()
        ln = (C.c_size_t * max(n, 1))()
        st = call(None, 0, C.byref(need), off, ln)
        if st not in (_lib.OK, _lib.ERR_DST_TOO_SMALL):
            self._check(st, "multi batch call")
        arena = np.empty(max(need.value, 1), dtype=np.uint8)
        if st == _lib.ERR_DST_TOO_SMALL:
            self._check(self.L.zipc_b200_multi_fetch(self.h, arena.ctypes.data, arena.size), "multi_fetch")
        return arena, off, ln

    def inflate_batch(self, items: Sequence, decompressed_sizes=None, crc_op: int = CK_NONE, adler_mode: int = ADLER_REF_COMPAT):
        vs = [_as_view(x) for x in items]
        n = len(vs)
        ptrs, lens = Context._ptr_arrays(vs)
        mo = (C.c_size_t * max(n, 1))()
        for i in range(n):
            d = None if decompressed_sizes is None else decompressed_sizes[i]
            mo[i] = SIZE_UNKNOWN if d is None else d
        ck = (C.c_uint32 * max(n, 1))()
        stt = (C.c_int * max(n, 1))()
        arena, off, ln = self._arena_call(
            lambda dst, cap, need, o, l: self.L.zipc_b200_multi_inflate_batch(self.h, crc_op, adler_mode, n, ptrs, lens, mo,
                                                                              dst, cap, need, o, l, ck, stt), n)
        return [(stt[i], arena[off[i]:off[i] + ln[i]], ck[i]) for i in range(n)]

    def deflate_batch(self, items: Sequence, level: str = "default", crc_op: int = CK_NONE, adler_mode: int = ADLER_REF_COMPAT):
        vs = [_as_view(x) for x in items]
        n = len(vs)
        ptrs, lens = Context._ptr_arrays(vs)
        ck = (C.c_uint32 * max(n, 1))()
        stt = (C.c_int * max(n, 1))()
        lv = LEVELS[level]
        arena, off, ln = self._arena_call(
            lambda dst, cap, need, o, l: self.L.zipc_b200_multi_deflate_batch(self.h, lv, crc_op, adler_mode, n, ptrs, lens, dst,
                                                                              cap, need, o, l, ck, stt), n)
        return [(stt[i], arena[off[i]:off[i] + ln[i]], ck[i]) for i in range(n)]


_default: Context | None = None


def default_context() -> Context:
    global _default
    if _default is None:
        _default = Context()
    return _default


def set_default_context(ctx: Context | None) -> None:
    global _default
    _default = ctx


# ---- Zipc_deflate.Crc_32 / Adler_32 ---------------------------------------------------------------
class _Checksum:
    @staticmethod
    def equal(a: int, b: int) -> bool:
        return (a & 0xFFFFFFFF) == (b & 0xFFFFFFFF)

    @classmethod
    def check(cls, expect: int, found: int):
        return Ok(None) if cls.equal(expect, found) else Error(_crc_error(expect, found), _lib.ERR_CHECKSUM, (expect, found))

    @staticmethod
    def pp(crc: int) -> str:
        return "%x" % crc


class Crc_32(_Checksum):
    """ZIP CRC-32 checksums (zipc_deflate.mli:24-48)."""

    @staticmethod
    def string(s, start: int = 0, len: int | None = None) -> int:
        return default_context().crc32(_slice(s, start, len))

    @staticmethod
    def strings(items: Iterable) -> list[int]:
        return default_context().crc32_batch(items)


class Adler_32(_Checksum):
    """Adler-32 checksums (zipc_deflate.mli:51-75).  mode: ADLER_REF_COMPAT reproduces the
    reference's signed Int32.rem bit for bit, ADLER_RFC1950 is the standard checksum."""

    @staticmethod
    def string(s, start: int = 0, len: int | None = None, mode: int = ADLER_REF_COMPAT) -> int:
        return default_context().adler32(_slice(s, start, len), mode)


# ---- decompression ---------------------------------------------------------------------------------
def _inflate_result(st, out, ck, crc_op):
    if st:
        return Error(strerror(st), st)
    data = out.tobytes()
    return Ok(data if crc_op == CK_NONE else (data, ck))


def inflate_batch(items, decompressed_sizes=None, crc_op: int = CK_NONE, adler_mode: int = ADLER_REF_COMPAT):
    res = default_context().inflate_batch(items, decompressed_sizes, crc_op, adler_mode)
    return [_inflate_result(st, out, ck, crc_op) for st, out, ck in res]


def inflate(s, decompressed_size: int | None = None, start: int = 0, len: int | None = None):
    """zipc_deflate.mli:79-90"""
    return inflate_batch([_slice(s, start, len)], [decompressed_size])[0]


def inflate_and_crc_32(s, decompressed_size: int | None = None, start: int = 0, len: int | None = None):
    """zipc_deflate.mli:92-96"""
    return inflate_batch([_slice(s, start, len)], [decompressed_size], CK_CRC32)[0]


def inflate_and_adler_32(s, decompressed_size: int | None = None, start: int = 0, len: int | None = None,
                         adler_mode: int = ADLER_REF_COMPAT):
    """zipc_deflate.mli:98-102"""
    return inflate_batch([_slice(s, start, len)], [decompressed_size], CK_ADLER32, adler_mode)[0]


def zlib_decompress_batch(items, decompressed_sizes=None, adler_mode: int = ADLER_REF_COMPAT):
    out = []
    for st, data, ex, fo in default_context().zlib_decompress_batch(items, decompressed_sizes, adler_mode):
        if st == _lib.ERR_CHECKSUM:
            out.append(Error(_crc_error(ex, fo), st, (ex, fo)))      # Error (Some (expect, found), msg)
        elif st == _lib.ERR_ZLIB_METHOD:
            out.append(Error("Unknown compression method (%d)" % fo, st))
        elif st:
            out.append(Error(strerror(st), st))                      # Error (None, msg)
        else:
            out.append(Ok((data.tobytes(), fo)))
    return out


def zlib_decompress(s, decompressed_size: int | None = None, start: int = 0, len: int | None = None,
                    adler_mode: int = ADLER_REF_COMPAT):
    """zipc_deflate.mli:104-118"""
    return zlib_decompress_batch([_slice(s, start, len)], [decompressed_size], adler_mode)[0]


# ---- compression -------------------------------------------------------------------------------------
def deflate_batch(items, level: str = "default", crc_op: int = CK_NONE, adler_mode: int = ADLER_REF_COMPAT):
    res = default_context().deflate_batch(items, level, crc_op, adler_mode)
    out = []
    for st, data, ck in res:
        if st:
            out.append(Error(strerror(st), st))
        else:
            out.append(Ok(data.tobytes() if crc_op == CK_NONE else (ck, data.tobytes())))
    return out


def deflate(s, level: str = "default", start: int = 0, len: int | None = None):
    """zipc_deflate.mli:128-137.  NB the reference's *implementation* defaults an omitted ?level to
    `Best (zipc_deflate.ml:817) although its documentation says `Default; we follow the docs."""
    return deflate_batch([_slice(s, start, len)], level)[0]


def crc_32_and_deflate(s, level: str = "default", start: int = 0, len: int | None = None):
    """zipc_deflate.mli:139-143"""
    return deflate_batch([_slice(s, start, len)], level, CK_CRC32)[0]


def adler_32_and_deflate(s, level: str = "default", start: int = 0, len: int | None = None,
                         adler_mode: int = ADLER_REF_COMPAT):
    """zipc_deflate.mli:145-149"""
    return deflate_batch([_slice(s, start, len)], level, CK_ADLER32, adler_mode)[0]


def zlib_compress_batch(items, level: str = "default", adler_mode: int = ADLER_REF_COMPAT):
    out = []
    for st, data, ad in default_context().zlib_compress_batch(items, level, adler_mode):
        out.append(Error(strerror(st), st) if st else Ok((ad, data.tobytes())))
    return out


def zlib_compress(s, level: str = "default", start: int = 0, len: int | None = None,
                  adler_mode: int = ADLER_REF_COMPAT):
    """zipc_deflate.mli:151-162"""
    return zlib_compress_batch([_slice(s, start, len)], level, adler_mode)[0]
